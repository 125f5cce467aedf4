/*
 * auvrrt.h -- C ABI of libauvrrt.so, the B200 (sm_100a) implementation of the RRT planning inner
 * loop of hmc-lair-shark-tracking/auv-sim.
 *
 * The reference has no FFI of its own: its boundary is the Python surface of
 * path_planning/rrt_dubins.py (class RRT) and path_planning/cost.py.  Each entry point below names
 * the reference function it replaces (file:line under /root/reference); INTEGRATION.md shows the
 * ctypes stub a maintainer adds on the reference side.
 *
 * Conventions
 *   - plain pointers and sizes, no torch types; every function returns an int status
 *     (AUVRRT_OK == 0) and auvrrt_last_error() returns a thread-local message for the last failure.
 *   - `precision`: AUVRRT_F32 = fast build (fp32 arithmetic, tolerance 1e-5 relative vs the fp64
 *     reference), AUVRRT_F64 = verification build (fp64, no FMA contraction, the reference's
 *     operation order; indices / booleans match the reference exactly).
 *   - Functions without a suffix take HOST buffers (always double / int32 / uint8 / uint64) and do
 *     their own host<->device copies on an internal stream.  Functions ending in `_dev` take DEVICE
 *     pointers whose floating type is float (AUVRRT_F32) or double (AUVRRT_F64) plus a cudaStream_t
 *     passed as void*; they enqueue work and return without synchronising.
 *   - An auvrrt_env_t owns reusable device / pinned scratch for the host-buffer planner entry, so one
 *     handle must not be used by two threads at once; separate handles are independent.
 *   - There is NO CPU fallback: without a CUDA device every compute entry fails with
 *     AUVRRT_ERR_CUDA.
 */
#ifndef AUVRRT_H
#define AUVRRT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AUVRRT_OK 0
#define AUVRRT_ERR_ARG 1
#define AUVRRT_ERR_CUDA 2
#define AUVRRT_ERR_UNSUPPORTED 3

#define AUVRRT_F32 0
#define AUVRRT_F64 1

/* per-query / per-edge status codes, mirroring the reference's uncaught exceptions */
#define AUVRRT_ST_OK 0
#define AUVRRT_ST_NO_PATH 1     /* TypeError at rrt_dubins.py:174 (opt_path is None) */
#define AUVRRT_ST_ZERO_DIV 2    /* ZeroDivisionError at rrt_dubins.py:270 / :281 */
#define AUVRRT_ST_KEY_ERROR 3   /* KeyError / IndexError at rrt_dubins.py:123-127 */
#define AUVRRT_ST_STREAM_END 4  /* explicit uniform stream exhausted */
#define AUVRRT_ST_OVERFLOW 5    /* a fixed-size output (chain / path) was too small */

typedef struct auvrrt_env auvrrt_env_t;

const char *auvrrt_last_error(void);
/* number of CUDA devices visible, 0 if none (never an error) */
int auvrrt_device_count(void);
/* kernels this library launched in this process since load (bench.py's gpu_launches) */
int64_t auvrrt_launch_count(void);

/* ---- world model ---------------------------------------------------------------------------
 * Replaces the Python objects RRT.__init__ keeps (rrt_dubins.py:26-49): obstacle circles in
 * obstacle_list order, the boundary polygon ring, habitats (cost.py:145), and the shark grid
 * {(t0,t1): {cell.bounds: p}} (createSharkGrid, rrt_dubins.py:612-630) flattened to
 * bins[T][2], cells[C][4] (minx,miny,maxx,maxy, dict order), probs[T][C].  Any count may be 0. */
int auvrrt_env_create(const double *circles, int K, const double *poly, int E,
                      const double *habitats, int H, const double *bins, int T,
                      const double *cells, int C, const double *probs, int device,
                      auvrrt_env_t **out);
void auvrrt_env_destroy(auvrrt_env_t *env);
/* The flattened world model exactly as the kernels read it (header + tables, csrc/env.cuh), built on the
 * host without touching a device: returns its size in bytes (-1 on a bad argument) and copies it to `out`
 * if cap is large enough.  For the CPU-only tests that check the classification grid and the shark-cell
 * index against the reference's exact predicates (rrt_dubins.py:530-549, cost.py:173-191). */
int64_t auvrrt_env_host_blob(const double *circles, int K, const double *poly, int E,
                             const double *habitats, int H, const double *bins, int T,
                             const double *cells, int C, const double *probs, int precision,
                             unsigned char *out, int64_t cap);

/* ---- RRT.get_closest_mps (rrt_dubins.py:505-513) ---------------------------------------------
 * nq queries against one tree of n nodes (SoA x[], y[]); strict <, lowest index wins ties;
 * compares sqrt(dx*dx + dy*dy) exactly as the reference does. */
int auvrrt_nn(const double *tree_x, const double *tree_y, int64_t n, const double *qx,
              const double *qy, int nq, int precision, int device, int32_t *out_idx);
int auvrrt_nn_dev(const void *tree_x, const void *tree_y, int64_t n, const void *qx, const void *qy,
                  int nq, int precision, void *scratch, int64_t scratch_bytes, int32_t *out_idx,
                  void *stream);
int64_t auvrrt_nn_scratch_bytes(int nq);

/* ---- RRT.steer, the random-arc rollout (rrt_dubins.py:237-295) --------------------------------
 * params = {dist_to_end, diff_max, freq, min_dist, velocity}.  Edge i starts at
 * parents[i] = (x, y, theta, traj_time_stamp, length) and consumes uniforms
 * u[uoff[i] .. uoff[i+1]) in the reference's order (SURVEY.md appendix A, steps 3-4).
 * Outputs: leaf[i] (same 5 fields), counts[i] = len(new.path) (parent included),
 * waypoints[i][k] = (x, y, theta, v, traj_time_stamp, length) for k < counts[i]-1 (wp_cap rows per
 * edge), used[i] = uniforms consumed, status[i]. */
int auvrrt_steer_arc(const double *parents, int64_t n, const double *u, const int64_t *uoff,
                     const double params[5], int precision, int device, double *leaf,
                     int32_t *counts, double *waypoints, int wp_cap, int32_t *used,
                     int32_t *status);

/* ---- six-word Dubins steer (named by the north star; rrt_dubins.py:238-251 is a commented-out
 * call into the absent PyPI `dubins` module -> parity unpinned, see DESIGN.md) -----------------
 * from/to = (x, y, theta); word in evaluation order LSL=0, LSR, RSL, RSR, RLR, LRL (255 = none);
 * seg = (t, p, q) in units of rho; length = rho (t+p+q); waypoints[i][k], k < W: samples at
 * s = k * length/(W-1) for k < W-1, then `to` itself. */
int auvrrt_steer_dubins(const double *from, const double *to, int64_t n, double rho, int W,
                        int precision, int device, uint8_t *word, double *seg, double *length,
                        double *waypoints);

/* ---- RRT.check_collision (rrt_dubins.py:530-549), True(1) = safe -----------------------------
 * Path i = points[off[i] .. off[i+1]) as (x, y).  Reproduces the running-minimum quirk
 * (:535-542) and strict-interior Point.within (:544-547, exact predicate in AUVRRT_F64).
 * An empty path with K > 0 raises ValueError in the reference: out_safe = 255. */
int auvrrt_collide(const auvrrt_env_t *env, const double *points, const int64_t *off, int64_t n,
                   int precision, uint8_t *out_safe);
/* check_collision_obstacle (rrt_dubins.py:551-556): single points, per-obstacle test */
int auvrrt_collide_points(const auvrrt_env_t *env, const double *points, int64_t n, int precision,
                          uint8_t *out_safe);

/* ---- cost.habitat_shark_cost_func (cost.py:145-207) ------------------------------------------
 * Path i = points[off[i] .. off[i+1]) as (x, y, traj_time_stamp) in the caller's order;
 * out[i] = (sum, c0, c1, c2).  bin_mask (T bytes, may be NULL) selects shark-grid bins
 * (the planner's filter, rrt_dubins.py:161-166).  n_habitats < 0 means all of env's habitats,
 * otherwise only the first n_habitats. */
int auvrrt_cost(const auvrrt_env_t *env, const double *points, const int64_t *off, int64_t n,
                const double *t_total, const double weights[3], const uint8_t *bin_mask,
                int n_habitats, int precision, double *out);
/* cost.habitat_shark_cost_point (cost.py:209-241): visited[H] bytes, time-bin row tb */
int auvrrt_cost_point(const auvrrt_env_t *env, const double *points, int64_t n,
                      const uint8_t *visited, int tb, const double weights[3], int precision,
                      double *out_sum);

/* ---- fused edge evaluation: steer + collide (+ cost), the config-4 micro-benchmark -----------
 * Dubins edges: one (from, to) pair per edge, W waypoints each.  Arc edges: edge i consumes the
 * counter stream of seed seeds[i] from position 0 (see auvrrt_stream_u).
 * The _cost variants (config 4 "cost on") also return, per edge, its share of
 * cost.habitat_shark_cost_func over the appended waypoints (cost.py:171-191): out_cost [n][3] =
 * sum of w3 * prob, number of waypoints inside a habitat, number of distinct habitats visited. */
int auvrrt_edges_dubins_dev(const auvrrt_env_t *env, const void *from, const void *to, int64_t n,
                            double rho, int W, int precision, uint8_t *out_safe, uint8_t *out_word,
                            void *out_length, void *stream);
int auvrrt_edges_arc_dev(const auvrrt_env_t *env, const void *parents, const uint64_t *seeds,
                         int64_t n, const double params[5], int precision, uint8_t *out_safe,
                         int32_t *out_counts, void *out_leaf, void *stream);
int auvrrt_edges_dubins(const auvrrt_env_t *env, const double *from, const double *to, int64_t n,
                        double rho, int W, int precision, uint8_t *out_safe, uint8_t *out_word,
                        double *out_length);
int auvrrt_edges_arc(const auvrrt_env_t *env, const double *parents, const uint64_t *seeds,
                     int64_t n, const double params[5], int precision, uint8_t *out_safe,
                     int32_t *out_counts, double *out_leaf);
/* Dubins edges with cost on: traj_time_stamp of waypoint k = arclength_k / velocity from 0 at `from`; out_cost as for the
 * arc edges, over waypoints 1..W-1 (waypoint 0 is the parent node, rrt_dubins.py:537 tests it, cost.py never sees it
 * as an appended point).  The world must have a boundary polygon (the culled kernel runs). */
int auvrrt_edges_dubins_cost_dev(const auvrrt_env_t *env, const void *from, const void *to, int64_t n,
                                 double rho, int W, double velocity, double w3, int precision,
                                 uint8_t *out_safe, uint8_t *out_word, void *out_length, void *out_cost,
                                 void *stream);
int auvrrt_edges_dubins_cost(const auvrrt_env_t *env, const double *from, const double *to, int64_t n,
                             double rho, int W, double velocity, double w3, int precision,
                             uint8_t *out_safe, uint8_t *out_word, double *out_length, double *out_cost);
int auvrrt_edges_arc_cost_dev(const auvrrt_env_t *env, const void *parents, const uint64_t *seeds,
                              int64_t n, const double params[5], double w3, int precision,
                              uint8_t *out_safe, int32_t *out_counts, void *out_leaf, void *out_cost,
                              void *stream);
int auvrrt_edges_arc_cost(const auvrrt_env_t *env, const double *parents, const uint64_t *seeds,
                          int64_t n, const double params[5], double w3, int precision,
                          uint8_t *out_safe, int32_t *out_counts, double *out_leaf, double *out_cost);

/* ---- the pre-generated sample sequence ------------------------------------------------------
 * u_k(seed): counter hash built from 32-bit multiplies (DESIGN.md section 3): position k is the word
 * hi:lo, hi = M32a((k+1) * 0x9E3779B9 + key_lo), lo = M32b((k+1) * 0x85EBCA77 + key_hi),
 * key = SplitMix64 finaliser of (seed+1) * golden; u = (word >> 11) * 2^-53, or (f32u != 0, what the
 * AUVRRT_F32 build consumes) its top 23 bits, (word >> 41) * 2^-23.  Host-side evaluation for
 * callers that replay it (e.g. to feed the unmodified reference). */
double auvrrt_stream_u(uint64_t seed, int64_t k, int f32u);

/* ---- RRT.exploring (rrt_dubins.py:92-176): batched independent planning queries --------------*/
typedef struct {
    int32_t iterations;      /* budget: steer calls per query (replaces the wall-clock budget) */
    int32_t mode;            /* 0: traj_time_stamp & plan_time (time-bin pick, :122-127)
                                1: plan_time False (get_random_mps + get_closest_mps, :136-139)
                                2: plan_time & not traj_time_stamp (get_closest_mps_time, :129-132,
                                   :515-528) on a simulated clock: steer call i happens at
                                   plan time i * max_plan_time / iterations
                                3: Dubins-RRT with best-parent selection -- NOT executed by the reference (its
                                   Dubins steer is a commented-out call into the absent PyPI `dubins` module,
                                   :238-251, under the nearest-node branch :136-141); the build's own definition,
                                   parity unpinned (DESIGN.md section 11): sample a state (:333-343), candidate
                                   parents = the nearest node + the nodes within near_radius (32 at most), per
                                   candidate a six-word Dubins path cut at dubins_eta with dubins_w waypoints,
                                   check_collision, path cost through that parent (cost.py:145-207); the
                                   cheapest safe candidate becomes the parent (warp min-reduction) */
    double bin_interval, v, max_traj_time;
    double dist_to_end, diff_max, freq, min_dist;   /* RRT.__init__ defaults 2, 0.5, 30; 0.5 (:141) */
    double weights[3];
    int32_t chain_cap;       /* max tree depth recorded per query (<= 255) */
    int32_t path_cap;        /* rows per query in out_path (0: no paths) */
    int32_t trace;           /* != 0: fill the per-iteration trace arrays (parity tests) */
    int32_t group;           /* lanes cooperating on one tree: 32 (default when 0), 16 or 8; 1 = one thread
                                per tree, the throughput planner for >= 10^5 queries (no in-kernel paths) */
    double max_plan_time;    /* the reference's wall-clock budget in seconds; only mode 2 reads it */
    /* mode 3 only (see above): turning radius, longest edge, neighbourhood radius, waypoints per edge (2..32,
     * the parent included) */
    double dubins_rho, dubins_eta, near_radius;
    int32_t dubins_w;
    int32_t reserved;
} auvrrt_plan_params_t;

/* one fixed-size record per query: the unit the multi-GPU gather moves */
typedef struct {
    int32_t status;          /* AUVRRT_ST_* */
    int32_t n_nodes;         /* len(mps_list) */
    int32_t best_node;       /* index into the tree of the optimal leaf, -1 if none */
    int32_t best_iter;       /* steer call that created it */
    int32_t depth;           /* edges from the root to best_node */
    int32_t n_path;          /* waypoints on the optimal path (len(path)) */
    int32_t n_cost_evals;    /* candidate leaves evaluated (t >= max_traj_time - 30) */
    int32_t n_waypoints;     /* sum of len(new.path) over all steer calls */
    int64_t n_uniforms;      /* stream positions consumed */
    int64_t n_primitives;    /* arc primitives drawn */
    double cost[4];          /* sum, c0, c1, c2 of the optimal path */
    double path_length;      /* "path length" of the result dict */
    double t_leaf;           /* traj_time_stamp of the optimal leaf */
} auvrrt_plan_record_t;

/* optional per-iteration trace, each [Q][iterations] (parity tests only) */
typedef struct {
    int32_t *parent; uint8_t *safe; int32_t *nwp; double *leaf /* [Q][I][5] */; int64_t *upos;
} auvrrt_plan_trace_t;

/* starts[Q][5] = (x, y, theta, traj_time_stamp, length); seeds[Q];
 * out_chain[Q][chain_cap]: stream positions of the steer calls root->leaf along the optimal path
 * (enough to re-create it with auvrrt_materialize); out_path[Q][path_cap][6] =
 * (x, y, theta, v, traj_time_stamp, length) in root->leaf order, i.e. result["path"][0].
 * out_chain may be NULL.  Status AUVRRT_ST_OVERFLOW is raised only where a chain buffer is passed: a plan
 * deeper than chain_cap is OVERFLOW with a chain and OK without one.  Records of plans with
 * depth <= chain_cap are the same either way.  Paths are written while walking the chain, so out_path
 * needs out_chain. */
int auvrrt_plan_batch(const auvrrt_env_t *env, const double *starts, const uint64_t *seeds,
                      int64_t Q, const auvrrt_plan_params_t *params, int precision,
                      auvrrt_plan_record_t *out_records, uint32_t *out_chain, double *out_path,
                      const auvrrt_plan_trace_t *trace);
/* device-resident variant: starts are float[Q][5] (F32) or double[Q][5] (F64); records / chain /
 * path / trace are device pointers (path rows in the precision's floating type; trace.leaf too).
 * workspace from auvrrt_plan_workspace_bytes(); nothing is synchronised.  out_path != NULL with
 * path_cap > 0 and out_chain == NULL is AUVRRT_ERR_ARG, and so is a workspace smaller than the
 * launch needs; either way nothing is written.
 * group 0 picks the kernel per call: one thread per tree for >= 32768 queries without paths
 * (mode != 3), else one warp per tree. */
int64_t auvrrt_plan_workspace_bytes(const auvrrt_env_t *env, const auvrrt_plan_params_t *params,
                                    int precision);
/* same, for a batch of at most Q queries (group == 1 sizes its workspace by the batch; group 0
 * covers every kernel a batch of at most Q queries can launch) */
int64_t auvrrt_plan_workspace_bytes_q(const auvrrt_env_t *env, const auvrrt_plan_params_t *params,
                                      int precision, int64_t Q);
int auvrrt_plan_batch_dev(const auvrrt_env_t *env, const void *starts, const uint64_t *seeds,
                          int64_t Q, const auvrrt_plan_params_t *params, int precision,
                          void *workspace, int64_t workspace_bytes,
                          auvrrt_plan_record_t *out_records, uint32_t *out_chain, void *out_path,
                          const auvrrt_plan_trace_t *trace, void *stream);

/* re-create optimal paths from (start, seed, chain) records, e.g. for the few winners after the
 * multi-GPU gather.  Same row layout as out_path; out_n_path[q] is the full row count even when it
 * exceeds path_cap (then only the first path_cap rows are written).  A depth of 0 gives the start
 * row alone.  Any depth[q] < 0 or > chain_cap (an OVERFLOW record) is AUVRRT_ERR_ARG, checked before
 * anything runs.  params->group must name the planner that made the chains, because the fp32 edge
 * evaluators of the group sizes round differently: 32 (or 0), 16, 8, or 1 for the thread-per-tree
 * planner -- which is also what group 0 ran for a batch of >= 32768 queries without paths. */
int auvrrt_materialize(const auvrrt_env_t *env, const double *starts, const uint64_t *seeds,
                       const uint32_t *chain, const int32_t *depth, int64_t Q,
                       const auvrrt_plan_params_t *params, int precision, double *out_path,
                       int32_t *out_n_path);

/* ---- the device end of a planning step: each mission's best plan and its path, all in HBM ------
 * auvrrt_plan_group: the group auvrrt_plan_batch(_dev) runs for a batch of Q queries -- 32, 16, 8 or
 * 1 -- where with_path says whether paths are written (out_path != NULL and path_cap > 0).  An
 * explicit group passes through; group 0 is 1 for Q >= 32768 without paths and mode != 3, else 32.
 * -1 (message set) for a bad group or mode 3 with group 1.  Host logic only: needs no device.  It is
 * the group auvrrt_materialize(_dev) needs to re-create the plans of that batch. */
int auvrrt_plan_group(const auvrrt_plan_params_t *params, int64_t Q, int with_path);
/* Each mission's best plan (RRT.exploring with replicas, rrt_dubins.py:169).  Device buffers: records
 * [Q], mission_off int64 [M + 1]; mission m is records [lo, hi) with lo = clamp(mission_off[m], 0, Q),
 * hi = clamp(mission_off[m + 1], lo, Q), so no offset reads out of bounds.  A record is eligible when
 * status == AUVRRT_ST_OK, depth >= 0 and cost[0] is not NaN (a plan made with a chain buffer and
 * deeper than chain_cap is OVERFLOW, not OK).  Among them the least cost[0] wins as floats compare
 * (-0.0 == +0.0), the lowest index on ties -- the reference's strict `<`.  out_best int64 [M]: the
 * global index of the winner, -1 if the mission has none; out_cost double [M]: its cost[0], +inf if
 * none.  Asynchronous on `stream`: no allocation, no synchronisation (it can be captured in a CUDA
 * graph).  Reads the first 64 bytes of each record (status, depth, cost[0]).  One kernel while
 * missions average at most 4096 records; past that 2 memsets and 3 kernels, each mission's records
 * split over CTAs. */
int auvrrt_plan_best_dev(const auvrrt_plan_record_t *records, int64_t Q, const int64_t *mission_off,
                         int64_t M, int64_t *out_best, double *out_cost, void *stream);
/* auvrrt_materialize on device buffers, through a pick list: output row m re-creates plan pick[m]
 * of the Q plans (starts [Q][5] in the precision's type, seeds [Q], records [Q], chain
 * [Q][chain_cap] of one auvrrt_plan_batch_dev call), with the depth of its record.  out_path
 * [M][path_cap][6] in the precision's type, out_n_path int32 [M] with the full row count (only the
 * first path_cap rows are written).  pick[m] == -1 (a mission without a plan) gives n_path 0; any
 * other pick outside [0, Q), or a depth outside [0, chain_cap] (e.g. an OVERFLOW record), gives
 * n_path -1; neither writes a row.  params->group must name the planner that made the chains: 32,
 * 16, 8 or 1 (auvrrt_plan_group of that batch); group 0 is AUVRRT_ERR_ARG.  Every argument error is
 * returned before anything is enqueued.  Rows equal auvrrt_materialize's for the same plans bit for
 * bit.  Asynchronous on `stream`, no allocation. */
int auvrrt_materialize_dev(const auvrrt_env_t *env, const void *starts, const uint64_t *seeds,
                           const auvrrt_plan_record_t *records, const uint32_t *chain, int64_t Q,
                           const int64_t *pick, int64_t M, const auvrrt_plan_params_t *params,
                           int precision, void *out_path, int32_t *out_n_path, void *stream);

/* ---- SharkOccupancyGrid.convert (sharkOccupancyGrid.py:47-71): shark tracks -> AUV-detection grids
 * SURVEY.md section 8(f) row N2, the producer of the cost function's probs[T][C] input.
 * cells: C polygons in cell_list order (vertices cell_xy[cell_off[c] .. cell_off[c+1]));
 * bounds = boundary.bounds; tracks: S sharks in dict order, points (x, y, traj_time_stamp) at
 * tracks[track_off[s] .. track_off[s+1]).  auvrrt_occupancy_dims gives T (createBinList, :307-320)
 * and the grid shape; out_grid[T][rows][cols] = resultArr (fp64, bit-identical to the reference).
 * The value of cell c in bin b (resultCell / createSharkGrid's CSV) is
 * out_grid[b][int((miny_c - bounds[1]) / cell_size)][int((minx_c - bounds[0]) / cell_size)]. */
int auvrrt_occupancy_dims(const double bounds[4], double cell_size, double bin_interval,
                          const double *tracks, const int64_t *track_off, int S, int *T, int *rows,
                          int *cols);
int auvrrt_occupancy_grid(const double *cell_xy, const int64_t *cell_off, int C,
                          const double bounds[4], double cell_size, double bin_interval,
                          double detect_range, const double *tracks, const int64_t *track_off,
                          int S, int device, double *out_grid, int64_t out_cap);

/* ---- the same grids from device-resident tracks, and a live world's shark-occupancy table ------
 * An auvrrt_occ_t is one SharkOccupancyGrid for fixed cells / bounds / cell_size / bin_interval /
 * detect_range (arguments as for auvrrt_occupancy_grid), with n_bins bins (b * bin_interval,
 * (b + 1) * bin_interval), at most max_sharks tracks and max_points points per call.  It owns the
 * cell tables, a candidate-cell index (built once, on the host) and its workspace, so a call
 * allocates nothing and synchronises nothing.
 *
 * auvrrt_occ_grid_dev: d_tracks [n_points][3] (x, y, traj_time_stamp) fp64 and d_track_off [S+1]
 * int64 on the device, S sharks in dict order (points in no [track_off[s], track_off[s+1]) are
 * skipped).  Writes d_grid [n_bins][rows][cols] fp64 if non-NULL; if env is non-NULL, replaces its
 * probs[T][C] (both precisions' tables) in place with probs[b][c] = grid[b][row_c][col_c], where
 * cell c of the world is polygon c of this handle, in cell_list order, as createSharkGrid lays
 * them out; if d_t_occ is non-NULL, writes createBinList's T for these tracks there (int32, as
 * auvrrt_occupancy_dims).  Bins b < min(n_bins, T) are bit-identical to bin b of
 * auvrrt_occupancy_grid for the same tracks; the caller reads *d_t_occ to know whether all are
 * covered.  Asynchronous on `stream`: memsets, then 4 kernels (3 when n_points == 0) plus 1 when
 * env is given.
 * Writing to env needs env's C == C, T == n_bins and bins exactly (b * bin_interval,
 * (b + 1) * bin_interval) in double, as createBinList builds them.  A mismatch, S < 1,
 * S > max_sharks or n_points > max_points is AUVRRT_ERR_ARG, checked before anything is enqueued,
 * so the world is left unchanged.
 * Ordering: work that reads the world on another stream -- including every host-buffer entry, which
 * runs on the world's internal stream -- must be ordered after the refresh by the caller (e.g. by
 * synchronising `stream`). */
typedef struct auvrrt_occ auvrrt_occ_t;
int auvrrt_occ_create(const double *cell_xy, const int64_t *cell_off, int C, const double bounds[4],
                      double cell_size, double bin_interval, double detect_range, int n_bins,
                      int max_sharks, int64_t max_points, int device, auvrrt_occ_t **out);
void auvrrt_occ_destroy(auvrrt_occ_t *o);
int auvrrt_occ_shape(const auvrrt_occ_t *o, int *T, int *rows, int *cols);
int auvrrt_occ_grid_dev(auvrrt_occ_t *o, const double *d_tracks, const int64_t *d_track_off, int S,
                        int64_t n_points, double *d_grid, auvrrt_env_t *env, int32_t *d_t_occ,
                        void *stream);
/* Replace a world's probs[T][C] (host table; device table, asynchronous on `stream`) or read it
 * back (precision AUVRRT_F64: the fp64 table; AUVRRT_F32: the fp32 table, widened).  The fp32
 * table holds each value rounded to nearest, as auvrrt_env_create stores it.  The same ordering
 * rule as above applies to auvrrt_env_set_probs_dev. */
int auvrrt_env_set_probs(auvrrt_env_t *env, const double *probs);
int auvrrt_env_set_probs_dev(auvrrt_env_t *env, const double *d_probs, void *stream);
int auvrrt_env_get_probs(const auvrrt_env_t *env, int precision, double *out);

/* ---- gym_rrt Planner_RRT: the goal-directed tree RRTEnv.step grows one node at a time ---------
 * (gym_rrt/envs/rrt_dubins.py:30-503, driven by gym_rrt/envs/rrt_env.py:182-247).  SURVEY.md 8(f) N1.
 * One handle holds Q independent episodes ("vectorised environments") resident in HBM: the tree
 * (mps_list), the (row, col, subsection) node lists of env_grid with occupied_grid_cells_array in
 * first-occupancy order, and optionally the dense node count of every sub-cell (the observation
 * RRTEnv.convert_rrt_grid_to_1D_num_of_nodes_only builds, rrt_env.py:265-277).
 * Sub-cells are addressed by the flat id (row * cols + col) * subsections + subsection, the index
 * RRTEnv.step receives as chosen_grid_cell_idx (rrt_env.py:206-222).
 * random.choice(seq) is seq[int(u * len(seq))] on the episode's sample sequence. */
typedef struct auvrrt_gym auvrrt_gym_t;

typedef struct {
    double x0, y0, x1, y1;        /* boundary_point[0], boundary_point[1] (rrt_dubins.py:47) */
    double exp_rate, dist_to_end, diff_max, freq;   /* :34 */
    double cell_side;             /* cell_side_length */
    int32_t subsections;          /* subsections_in_cell */
    int32_t node_cap;             /* nodes one episode may hold, start included (steps + 1 is enough) */
    int32_t track_counts;         /* 1: keep the dense per-sub-cell node counts */
    int32_t reserved;
} auvrrt_gym_params_t;

typedef struct {
    int32_t status;               /* AUVRRT_ST_*; an episode with status != 0 no longer steps */
    int32_t done;                 /* generate_one_node returned True: a collision-free goal arc exists */
    int32_t steps;                /* generate_one_node calls so far */
    int32_t n_nodes;              /* len(mps_list) */
    int32_t n_occupied;           /* len(occupied_grid_cells_array) */
    int32_t last_parent;          /* mps_list index steered from in the last step, -1: empty cell, nothing done */
    int32_t last_accepted;        /* the last step appended its node (valid_new_node) */
    int32_t last_nwp;             /* arc primitives the last steer kept (len(new_node.path) - 1) */
    int32_t last_uniforms;        /* uniforms generate_one_node consumed in the last step */
    int32_t n_path;               /* len(path) of generate_final_course when done, else 0 */
    int64_t n_uniforms;           /* sample-sequence position */
    double cand[4];               /* the last steered node: x, y, theta, traj_time_stamp */
    double arc_length;            /* final_node.length (rrt_dubins.py:409) when done */
} auvrrt_gym_record_t;            /* 88 bytes */

int auvrrt_gym_create(const double *circles, int K, const auvrrt_gym_params_t *params, int64_t Q,
                      int precision, int device, auvrrt_gym_t **out);
void auvrrt_gym_destroy(auvrrt_gym_t *g);
/* discretize_env (rrt_dubins.py:77-93): rows = int(height) // int(cell_side), cols likewise */
int auvrrt_gym_grid_shape(const auvrrt_gym_t *g, int *rows, int *cols);
/* Planner_RRT.__init__ for every episode: starts [Q][3] = x, y, theta; goals [Q][2]; seeds [Q] */
int auvrrt_gym_reset(auvrrt_gym_t *g, const double *starts, const double *goals, const uint64_t *seeds);
/* Planner_RRT.__init__ for the episodes with d_mask[q] != 0 (d_mask == NULL: all, as auvrrt_gym_reset), on device
 * buffers d_starts [Q][3], d_goals [Q][2] (double), d_seeds [Q]; rows of episodes outside the mask are not read.
 * Asynchronous on `stream`.  Clears only what the episode's previous tree occupied.  A masked call needs one
 * earlier full reset of the handle (AUVRRT_ERR_ARG otherwise). */
int auvrrt_gym_reset_dev(auvrrt_gym_t *g, const uint8_t *d_mask, const double *d_starts, const double *d_goals,
                         const uint64_t *d_seeds, void *stream);
/* n_steps generate_one_node calls per episode, stopping early at done.  actions == NULL: the cell
 * is drawn with random.choice(occupied_grid_cells_array) (Planner_RRT.planning, :157-196);
 * else actions[Q] flat sub-cell ids (n_steps must be 1): RRTEnv.step; an empty cell does nothing.
 * full_candidates != 0 keeps steering after a collision so that cand[] is the reference's new_node
 * even for rejected steps (parity tests); 0 stops at the first colliding waypoint.
 * out_records [Q] may be NULL. */
int auvrrt_gym_step(auvrrt_gym_t *g, const int32_t *actions, int n_steps, int full_candidates,
                    auvrrt_gym_record_t *out_records);
/* same on device buffers (d_actions int32[Q] or NULL, d_records [Q] or NULL), asynchronous on `stream` */
int auvrrt_gym_step_dev(auvrrt_gym_t *g, const int32_t *d_actions, int n_steps, int full_candidates,
                        auvrrt_gym_record_t *d_records, void *stream);
/* episode q's tree: nodes [n][4] = x, y, theta, traj_time_stamp; parents [n]; cells [n] flat
 * sub-cell id or -1; occupied [n_occupied] in first-occupancy order.  Any pointer may be NULL. */
int auvrrt_gym_tree(const auvrrt_gym_t *g, int64_t q, int32_t cap, double *nodes, int32_t *parents,
                    int32_t *cells, int32_t *occupied, int32_t *n_nodes, int32_t *n_occupied);
/* dense node counts of episodes [q0, q0 + nq): out [nq][rows * cols * subsections] uint16;
 * needs track_counts.  auvrrt_gym_counts_dev returns the resident device array [Q][...]. */
int auvrrt_gym_counts(const auvrrt_gym_t *g, int64_t q0, int64_t nq, uint16_t *out);
const uint16_t *auvrrt_gym_counts_dev(const auvrrt_gym_t *g);
/* generate_final_course (rrt_dubins.py:318-328) of a done episode: path [n][3] = x, y, theta from
 * the goal arc's end back to the start (the reference does not reverse it). */
int auvrrt_gym_path(const auvrrt_gym_t *g, int64_t q, int32_t cap, double *path, int32_t *n_path);

/* ---- fixed-length lattice A* with the shark-occupancy cost (SURVEY.md 8(f) N4) -----------------
 * path_planning/astar_fixLenSOG.py: class astar (:114-141), method astar (:551-657) and its helpers
 * within_bounds (:178-203), collision_free (:205-221), curr_neighbors (:248-266), findCurrSOG
 * (:454-468), get_cell_prob (:486-510), get_top_n_prob (:520-536), smoothPath / Walkable (:223-246,
 * :416-452).  Deterministic; fp64 with separately rounded operations, bit-identical to the
 * reference.  One warp per query, Q independent queries (start, length limit, weights, velocity)
 * against one world.  Inputs the reference obtains through third parties are passed in: the
 * boundary centroid (shapely, :191) and the cell bounds after Python's round(v, 2) (:494-495). */
typedef struct auvrrt_astar_env auvrrt_astar_env_t;

typedef struct {
    double start[2];              /* self.start */
    double path_len_limit;        /* pathLenLimit */
    double weights[4];            /* w1..w4 (w1 is unused by the reference) */
    double velocity;              /* AUV_velocity */
} auvrrt_astar_query_t;           /* 64 bytes */

typedef struct {
    int32_t status;               /* AUVRRT_ST_OK; NO_PATH: the open list ran empty (astar returns None);
                                     KEY_ERROR: AttributeError (no time bin holds the time stamp, :489),
                                     TypeError (no cell holds the point, :602), IndexError (:532, :419,
                                     :652); OVERFLOW: node_cap / path_cap too small */
    int32_t n_expanded;           /* nodes taken off the open list */
    int32_t n_nodes;              /* nodes ever put on the open list (start included) */
    int32_t n_path;               /* len(result["node"]) */
    int32_t n_smooth;             /* result["path length"] = len(smoothPath(...)) */
    int32_t reserved;
    double cost;                  /* result["cost"] = cost of the last node */
    double path_len;              /* its pathLen */
} auvrrt_astar_record_t;          /* 40 bytes */

int auvrrt_astar_env_create(const double *circles, int K, const double *boundary, int E,
                            const double centroid[2], const double *habitats, int H,
                            const double *bins, int T, const double *cells_rounded, int C,
                            const double *probs, int device, auvrrt_astar_env_t **out);
void auvrrt_astar_env_destroy(auvrrt_astar_env_t *env);
/* paths [Q][path_cap][6] rows start -> goal = x, y, pathLen, time_stamp, cost, f (result["node"]);
 * keep [Q][path_cap] = 1 where smoothPath keeps the trajectory point (result["path"]);
 * expand_order NULL or [Q][node_cap] node ids in the order they left the open list;
 * node_xy NULL or [Q][node_cap][2].  paths / keep may be NULL (records only). */
int auvrrt_astar_batch(auvrrt_astar_env_t *env, const auvrrt_astar_query_t *queries, int64_t Q,
                       int32_t node_cap, int32_t path_cap, auvrrt_astar_record_t *records,
                       double *paths, uint8_t *keep, int32_t *expand_order, double *node_xy);
/* device buffers; workspace of auvrrt_astar_workspace_bytes(Q, node_cap) bytes; asynchronous on `stream` */
int64_t auvrrt_astar_workspace_bytes(int64_t Q, int32_t node_cap);
int auvrrt_astar_batch_dev(auvrrt_astar_env_t *env, const auvrrt_astar_query_t *d_queries, int64_t Q,
                           int32_t node_cap, int32_t path_cap, void *d_workspace,
                           int64_t workspace_bytes, auvrrt_astar_record_t *d_records, double *d_paths,
                           uint8_t *d_keep, int32_t *d_expand_order, double *d_node_xy, void *stream);

/* FP32 FFMA issue-rate calibration kernel for the roofline denominator: runs `iters` dependent
 * FFMA chains on every lane of a full grid and returns achieved FLOP/s (FMA = 2). */
int auvrrt_calibrate_fp32(int device, int iters, double *out_flops, double *out_ms);

#ifdef __cplusplus
}
#endif
#endif /* AUVRRT_H */
