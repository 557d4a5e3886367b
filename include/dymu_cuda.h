/*
 * dymu_cuda.h -- C ABI of the B200 (sm_100a) device library for DyMu's
 * total-cost propagation hot path (libdymu_cuda.so).
 *
 * The reference (ESA-PRL/planning-path_planning) is a single C++ class with no
 * FFI of its own; the host-side drop-in class in
 * planning-path_planning_b200/src/DyMu.hpp keeps that class interface and calls
 * ONLY the functions below.  Every entry point names the reference code whose
 * arithmetic it reproduces ("G.cpp" = src/DyMu_GlobalPathPlanning.cpp,
 * "L.cpp" = src/DyMu_LocalPathRepairing.cpp, "H.hpp" = src/DyMu.hpp).
 *
 * Conventions
 *  - extern "C", opaque context, plain pointers and sizes, no C++/torch types.
 *  - every call returns DYMU_OK (0) or a negative DYMU_ERR_* code; the text of
 *    the last error is available from dymu_last_error().  Nothing throws.
 *  - host matrices are row-major [j][i] with `ld` doubles per row (ld >= nx).
 *  - all arithmetic is IEEE fp64 without FMA contraction, in the reference's
 *    expression order.
 *  - a context is bound to one CUDA device and one stream; not thread-safe
 *    (the reference class is not either, H.hpp:397-609); use one context per
 *    GPU / per host thread.
 *  - there is no CPU fallback: without a CUDA device dymu_create fails.
 */
#ifndef DYMU_CUDA_H
#define DYMU_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dymu_ctx dymu_ctx;

#define DYMU_OK 0
#define DYMU_ERR_CUDA (-1)      /* a CUDA runtime call failed */
#define DYMU_ERR_ARG (-2)       /* invalid argument */
#define DYMU_ERR_STATE (-3)     /* call sequence error (e.g. solve before cost map) */
#define DYMU_ERR_NOCONV (-4)    /* iteration cap reached before convergence */
#define DYMU_ERR_CAPACITY (-5)  /* output buffer / local window too small */
#define DYMU_ERR_NODEVICE (-6)  /* no usable CUDA device */

/* fp64 planes of the global layer (globalNode fields, H.hpp:69-108) */
#define DYMU_PLANE_ELEVATION 0
#define DYMU_PLANE_SLOPE 1
#define DYMU_PLANE_RAW_COST 2
#define DYMU_PLANE_COST 3
#define DYMU_PLANE_HAZARD_DENSITY 4
#define DYMU_PLANE_TRAFFICABILITY 5
#define DYMU_PLANE_TOTAL_COST 6 /* slot 0; other slots through dymu_download_total_cost */
#define DYMU_PLANE_CEFF 7       /* global_res*cost*(2+hazard-trafficability), obstacle = +inf */
/* directional costs a(x->m) of the anisotropic solve, toward the neighbour at i-1, i+1, j-1,
 * j+1 (see dymu_set_anisotropy).  Read-only; they exist only while anisotropy is on. */
#define DYMU_PLANE_DIRCOST_XM 8
#define DYMU_PLANE_DIRCOST_XP 9
#define DYMU_PLANE_DIRCOST_YM 10
#define DYMU_PLANE_DIRCOST_YP 11
/* distance in metres from a cell to the nearest obstacle cell, +inf beyond radius + margin (see
 * dymu_set_obstacle_clearance).  Read-only; it exists only while obstacle clearance is on. */
#define DYMU_PLANE_CLEARANCE 12
/* byte / word planes */
#define DYMU_PLANE_U8_OBSTACLE 0
#define DYMU_PLANE_U8_LOCMODE 1 /* index into locomotion_modes, 255 = "DONT_CARE" */

/* read-back transforms */
#define DYMU_XFORM_NONE 0
#define DYMU_XFORM_INF_TO_MINUS1 1   /* getTotalCostMatrix, G.cpp:799-811 */
#define DYMU_XFORM_EFFECTIVE_COST 2  /* getGlobalCostMatrix, G.cpp:815-829 (on DYMU_PLANE_COST) */

typedef struct dymu_solve_stats
{
    uint32_t outer_iterations;  /* grid-wide sweep phases of the tile FIM */
    uint32_t converged;         /* 1 if the active list drained */
    uint64_t tile_activations;  /* tiles loaded, relaxed in shared memory and stored */
    uint64_t cell_updates;      /* evaluations of the upwind update (G.cpp:500-546) */
    uint64_t cells_reached;     /* cells with finite total cost (filled by dymu_count_reached) */
    uint64_t tiles_deferred;    /* list entries carried over by the priority band */
    uint64_t inner_iterations;  /* shared-memory sweeps summed over tile activations */
    float kernel_ms;            /* device time of the solve kernel(s), CUDA events */
    float reset_ms;             /* device time of the total-cost reset */
    uint32_t goal_obstacle;     /* goals that sit on an obstacle cell and were therefore not seeded
                                   ("The goal is not valid", G.cpp:370-374) */
    uint32_t tiles_delivered_early; /* direct delivery (dymu_set_total_cost_export): tiles stored to the
                                       caller's matrix while the solve was still running ... */
    uint64_t cells_written;     /* cells whose value was stored back to the plane (8 B each) */
    uint32_t tiles_delivered_late;  /* ... and tiles stored after the last phase */
    uint32_t reserved_;
} dymu_solve_stats;

/* ---- context ---------------------------------------------------------- */

/* Global layer allocation.  Replaces initGlobalLayer's per-node `new`
 * (G.cpp:39-104) with SoA device planes.  device < 0 = current device. */
int dymu_create(int device, uint32_t nx, uint32_t ny, double global_res, double local_res,
                dymu_ctx** out);
int dymu_destroy(dymu_ctx* ctx);
const char* dymu_last_error(const dymu_ctx* ctx);
/* The CUDA stream all work of this context is issued on (cudaStream_t). */
void* dymu_stream(dymu_ctx* ctx);
int dymu_synchronize(dymu_ctx* ctx);
/* Number of kernel launches issued by this context so far. */
uint64_t dymu_launch_count(const dymu_ctx* ctx);
/* Device-side timing on the context's stream: record user event `which` (0..7) and read
 * the elapsed milliseconds between two recorded events (synchronises on event b). */
int dymu_event_record(dymu_ctx* ctx, int which);
int dymu_event_elapsed_ms(dymu_ctx* ctx, int a, int b, float* ms);
/* Self-test: compares the solver's branch-free square root with the IEEE sqrt on n
 * pseudo-random positive normal doubles; *mismatches must come back 0. */
int dymu_selftest_sqrt(dymu_ctx* ctx, uint64_t n, uint64_t seed, uint64_t* mismatches,
                       double* first_bad);
/* Times the streaming stencil kernels of the path once each on the resident planes (CUDA
 * events on the context's stream).  ms[0..5] = total-cost reset (k_fill_f64), C_eff build
 * (k_ceff), read-back transform (k_readback), setCostMap mask (k_set_cost_map), slope +
 * nominal cost (k_slope_nominal; -1 if computeCostMap was never called), smoothing
 * (k_smooth_cost on a scratch copy).  All are idempotent on the context's state. */
int dymu_time_stencils(dymu_ctx* ctx, float ms[6]);
/* Tile geometry of the solver: tile edge (cells), padded pitch (doubles per row). */
int dymu_geometry(const dymu_ctx* ctx, uint32_t* tile, uint32_t* pitch, uint32_t* rows);

/* ---- plane I/O ---------------------------------------------------------- */
int dymu_upload_plane(dymu_ctx* ctx, int plane, const double* host, size_t ld);
int dymu_download_plane(dymu_ctx* ctx, int plane, double* host, size_t ld, int xform);
int dymu_download_plane_u8(dymu_ctx* ctx, int plane, uint8_t* host, size_t ld);
/* rectangle [i0,i0+w) x [j0,j0+h) of a plane <-> dense host buffer (w*h doubles) */
int dymu_read_rect(dymu_ctx* ctx, int plane, uint32_t i0, uint32_t j0, uint32_t w, uint32_t h,
                   double* host);
int dymu_write_rect(dymu_ctx* ctx, int plane, uint32_t i0, uint32_t j0, uint32_t w, uint32_t h,
                    const double* host);
int dymu_read_rect_u8(dymu_ctx* ctx, int plane, uint32_t i0, uint32_t j0, uint32_t w, uint32_t h,
                      uint8_t* host);
/* Raw device pointer of a plane (for callers that fill planes on the device). */
int dymu_plane_device_ptr(dymu_ctx* ctx, int plane, void** dptr, size_t* pitch_elems);

/* ---- cost map ------------------------------------------------------------- */
/* setCostMap, G.cpp:109-126: cost copy; cost <= 0 => obstacle, trafficability 0,
 * hazard_density 1.  `host` may be NULL if DYMU_PLANE_COST was already filled. */
int dymu_set_cost_map(dymu_ctx* ctx, const double* host, size_t ld);
/* computeCostMap, G.cpp:145-308: slope (G.cpp:186-210), nominal cost from the
 * [terrain][locomotion][slope] table incl. obstacle marking (G.cpp:217-293),
 * 5-point smoothing seeded with the previous cost (G.cpp:297-308).
 * elevation/terrain may be NULL if already resident: a terrain map staged by
 * dymu_upload_terrain is consumed by the next call; after that the terrain classes stay in
 * HBM, so a call with both NULL rebuilds the cost map from a new table alone (the
 * updateCost -> computeCostMap loop of CoRa, G.cpp:956-993, without re-sending the DEM). */
int dymu_compute_cost_map(dymu_ctx* ctx, const double* cost_lut, int n_lut, const double* slopes,
                          int n_slopes, int n_locs, const double* elevation, size_t ld_e,
                          const double* terrain, size_t ld_t);
int dymu_upload_terrain(dymu_ctx* ctx, const double* terrain, size_t ld);

/* ---- slope anisotropy (an extension; the reference's update is isotropic) -------------
 * n >= 2 pairs (theta_deg[k], factor[k]): signed slope angle in degrees, strictly ascending,
 * positive = uphill in the direction of travel; factor finite and > 0.  f(theta) is piecewise
 * linear in the table and clamped at both ends:
 *     f = factor[k] + (factor[k+1]-factor[k]) * ((theta-theta_deg[k]) / (theta_deg[k+1]-theta_deg[k]))
 * for theta_deg[k] <= theta < theta_deg[k+1].  For a cell x and its 4-neighbour m
 *     theta(x->m) = atan((elev[m]-elev[x]) / global_res) * (180/pi)
 *     a(x->m)     = C_eff(x) * f(theta(x->m))      (C_eff: DYMU_PLANE_CEFF; +inf toward outside)
 * (with obstacle clearance on, C_eff is the clearance-adjusted one)
 * and the total-cost update of x is the smallest of the four one-sided values T[m] + a(x->m)
 * and, for each pair (h in {i-1,i+1}, v in {j-1,j+1}) with -a_h < T_h - T_v < a_v, the root
 *     ((a_v^2*T_h + a_h^2*T_v) + (a_h*a_v)*sqrt((a_h^2+a_v^2) - d^2)) / (a_h^2+a_v^2),  d = T_h-T_v.
 * The descent scales the per-axis differences of gradientNode by 1/a^2 of the move against
 * them and normalises (DESIGN.md section 10).  While on, dymu_solve_total_cost,
 * dymu_solve_incremental (always a full solve), dymu_plan_streamed (upload first, then the full
 * solve), the path extraction and dymu_batch_solve are anisotropic; dymu_solve_start,
 * dymu_solve_advance and dymu_dd_solve return DYMU_ERR_STATE.  n = 0 switches it off and frees
 * the directional-cost planes; any other malformed table is DYMU_ERR_ARG. */
#define DYMU_ANISO_MAX 64
int dymu_set_anisotropy(dymu_ctx* ctx, const double* theta_deg, const double* factor, int n);

/* ---- obstacle clearance (an extension; the reference plans for a point) ---------------------
 * radius, margin, penalty: finite, >= 0, metres (penalty: dimensionless).  With g = global_res and
 * R = floor((radius + margin) / g) <= DYMU_CLEARANCE_MAX_CELLS, let s(x) be the smallest
 * di*di + dj*dj over obstacle cells (i+di, j+dj) with |di| <= R and |dj| <= R (cells outside the grid
 * are not obstacles).  The clearance is d(x) = sqrt(s) * g, +inf when there is no such obstacle or
 * d > radius + margin (= distance_transform_edt of the free cells times g, cut off there).  With c the
 * plain cost term (DYMU_PLANE_CEFF without clearance), C_eff becomes
 *     +inf                                                 on obstacles and for d <= radius (lethal ring)
 *     c * (1.0 + penalty * ((radius + margin - d) / margin))  for radius < d < radius + margin
 *     c                                                    otherwise
 * Lethal-ring cells are never propagation targets, like obstacles, but the obstacle plane stays as it
 * is.  So a goal inside the ring is not a valid goal: the solve still seeds it (only goals on obstacle
 * cells are refused), but the planner class rejects it as it rejects a goal on an obstacle.  A start
 * inside the ring has no finite total cost, like a start on an obstacle.  Every
 * solve reads the adjusted C_eff: dymu_solve_total_cost (any slot count), dymu_solve_incremental
 * (still incremental), dymu_solve_start / _advance on a whole grid, dymu_batch_solve, direct delivery,
 * the path extraction and, through the directional costs, slope anisotropy.  dymu_plan_streamed and a
 * streamed dymu_set_cost_map_begin complete the upload first and then run the full solve (clearance
 * near a seam needs rows that have not arrived yet).  dymu_dd_solve returns DYMU_ERR_STATE when any
 * strip has clearance on (a strip cannot see obstacles across a cut); a phase-bounded solve on a
 * strip sees only that strip's obstacles.  The clearance plane is rebuilt only when the obstacle
 * plane changed (dymu_set_cost_map, dymu_compute_cost_map, a streamed upload); changes of cost,
 * hazard_density or trafficability only re-run the C_eff pass.  radius == 0 && margin == 0 switches
 * it off and frees its planes; a negative, NaN or infinite value, or R > DYMU_CLEARANCE_MAX_CELLS, is
 * DYMU_ERR_ARG.  While it is off, DYMU_PLANE_CLEARANCE is an unknown plane (DYMU_ERR_ARG).  Any
 * change marks the resident total-cost map as stale. */
#define DYMU_CLEARANCE_MAX_CELLS 128
int dymu_set_obstacle_clearance(dymu_ctx* ctx, double radius, double margin, double penalty);

/* ---- total-cost solve -------------------------------------------------------- */
/* Number of independent total-cost planes ("slots") for batched goal queries. */
int dymu_reserve_slots(dymu_ctx* ctx, uint32_t n_slots);
/* computeEntireTotalCostMap / computeTotalCostMap, G.cpp:364-568: fixed point of the
 * first-order upwind update propagateGlobalNode (G.cpp:500-546) with T(goal) = 0, by a
 * tiled Fast Iterative Method.  n_goals independent problems are solved concurrently,
 * problem q writing slot q.  `stats` may be NULL or point to n_goals entries
 * (aggregate numbers are reported in stats[0]). */
int dymu_solve_total_cost(dymu_ctx* ctx, uint32_t n_goals, const uint32_t* goal_i,
                          const uint32_t* goal_j, dymu_solve_stats* stats);
/* Phase-bounded variants for pipelined domain decomposition (one GPU per row strip of a grid
 * too large or too slow for one GPU).  The propagation of computeEntireTotalCostMap
 * (G.cpp:443-468) is advanced by at most `max_phases` solver phases per call; the pending work
 * lists stay on the device between calls, stats->converged tells whether anything is left.
 *   dymu_solve_start    reset slot 0, seed the goal, run <= max_phases
 *   dymu_solve_advance  merge the tiles covering the row ranges (halo rows whose values were
 *                       just lowered by dymu_import_rows_min_key; n_ranges may be 0) into the
 *                       pending work with priority `seed_key` (the smallest lowered value) and
 *                       run <= max_phases more.  A strip without the goal starts with
 *                       dymu_reset_total_cost and its first import.  When nothing is pending
 *                       (after a converged solve or dymu_reset_total_cost), the call wakes the
 *                       tiles of `ranges` on a clean work list. */
int dymu_solve_start(dymu_ctx* ctx, uint32_t goal_i, uint32_t goal_j, uint32_t max_phases,
                     dymu_solve_stats* stats);
int dymu_solve_advance(dymu_ctx* ctx, const uint32_t* ranges, uint32_t n_ranges, double seed_key,
                       uint32_t max_phases, dymu_solve_stats* stats);
/* computeEntireTotalCostMap (G.cpp:443-468) again after cost, hazard_density or trafficability
 * changed a little -- the local layer's feedback (L.cpp:264-274, 388-394) -- without starting
 * over: cells whose cost term C (G.cpp:527-528) went up are found, everything that may have been
 * computed from them (reachable along strictly increasing total cost) goes back to +inf, and only
 * that region plus the tiles of cells whose C went down are propagated again.  Same fixed point
 * as dymu_solve_total_cost.  Needs the resident map of slot 0 to be the converged solve of the
 * same goal; otherwise, or when the invalidated cone does not fit its buffer (a quarter of the
 * plane), it IS dymu_solve_total_cost.  cells_invalidated (optional): cells reset, UINT64_MAX
 * when a full solve ran. */
int dymu_solve_incremental(dymu_ctx* ctx, uint32_t goal_i, uint32_t goal_j, dymu_solve_stats* stats,
                           uint64_t* cells_invalidated);
/* setCostMap (G.cpp:109-126) without waiting for the copy: the rows around `first_row` (the
 * goal's row; >= ny = middle) are sent first on the copy stream -- three parts: +-128 rows, then
 * +-max(256, ny/8), then the rest -- and the call returns at once.  The
 * next dymu_solve_total_cost with a single goal inside those first rows starts on them while the
 * rest is still arriving (see dymu_plan_streamed); every other entry point first completes the
 * upload and the obstacle bookkeeping, exactly as dymu_set_cost_map would have.  `cost_host` must
 * stay valid and unchanged until that next call returns, and should be pinned memory. */
int dymu_set_cost_map_begin(dymu_ctx* ctx, const double* cost_host, size_t ld, uint32_t first_row);
/* setCostMap (G.cpp:109-126) + computeEntireTotalCostMap (G.cpp:443-468) for a cost map that is
 * still in host memory, with the upload hidden behind the solve: the rows around the goal go
 * first, the solve starts on them with everything else impassable (C_eff = +inf); whenever the
 * next part of the upload has arrived the solve kernel hands back, the new rows are opened, the
 * tiles along the two seams re-activated and the solve goes on from its work lists.
 * first_phases == 0: the kernel hands back when the copy engine reports the part (a device word
 * written behind it in stream order); first_phases > 0 (or the environment variable
 * DYMU_STREAM_PHASES): after first_phases / 2 * first_phases solver phases instead.  Same fixed
 * point as dymu_set_cost_map + dymu_solve_total_cost.  `cost_host` should be pinned memory. */
int dymu_plan_streamed(dymu_ctx* ctx, const double* cost_host, size_t ld, uint32_t goal_i,
                       uint32_t goal_j, uint32_t first_phases, dymu_solve_stats* stats);
/* resetTotalCostMap (G.cpp:473-485) without seeding a goal: every slot-0 value = +inf. */
int dymu_reset_total_cost(dymu_ctx* ctx);
/* Halo exchange for row-strip domain decomposition.  Rows are dense (nx doubles each).
 * `device_ptr` != 0: dst/src is device memory of this GPU, otherwise host memory.
 * import takes the element-wise minimum with the resident rows, reports whether any
 * value decreased and sets *min_lowered = the smallest value that replaced a larger one
 * (+inf if none). */
int dymu_export_rows(dymu_ctx* ctx, uint32_t slot, uint32_t j0, uint32_t n_rows, double* dst,
                     int device_ptr);
int dymu_import_rows_min_key(dymu_ctx* ctx, uint32_t slot, uint32_t j0, uint32_t n_rows,
                             const double* src, int device_ptr, int* changed, double* min_lowered);
int dymu_count_reached(dymu_ctx* ctx, uint32_t slot, uint64_t* n_finite);
/* CLOSED-set emulation of the early stop in computeTotalCostMap (G.cpp:390): returns
 * T_stop = max over the start node and its 4 neighbours; cells with T <= T_stop are the
 * ones the reference would have CLOSED. */
int dymu_stop_threshold(dymu_ctx* ctx, uint32_t slot, uint32_t start_i, uint32_t start_j,
                        double* t_stop);
int dymu_download_total_cost(dymu_ctx* ctx, uint32_t slot, double* host, size_t ld, int xform);
/* getTotalCostMatrix (G.cpp:799-811) overlapped with getPath (G.cpp:589-611): _begin forks a
 * copy stream behind everything queued so far and returns at once; the caller may run
 * dymu_extract_global_path meanwhile, but nothing that changes the total-cost plane or
 * downloads another transformed plane; _end waits for the copy.  `host` should be pinned
 * memory, otherwise the copy is not asynchronous. */
int dymu_download_total_cost_begin(dymu_ctx* ctx, uint32_t slot, double* host, size_t ld, int xform);
/* Direct delivery of getTotalCostMatrix (G.cpp:799-811): from now on every full single-goal solve
 * (dymu_solve_total_cost, dymu_plan_streamed, dymu_solve_incremental when it solves from scratch)
 * stores the total-cost matrix into `host` (row stride `ld` doubles) itself -- each tile as soon as
 * the wave front is past it, the rest right after the last phase on the copy stream (it is
 * complete when dymu_download_total_cost_end, dymu_download_total_cost or dymu_synchronize return) -- instead of
 * leaving it to a copy afterwards; a later dymu_download_total_cost[_begin] with the same host / ld / xform then
 * has nothing left to copy.  `host` must be page-locked memory the device can write to
 * (cudaHostAlloc / cudaHostRegister, e.g. a torch pinned tensor); otherwise nothing is set up and
 * *direct comes back 0 (not an error).  The buffer is written during the solve and is only
 * meaningful after a solve that returned DYMU_OK.  host == NULL switches it off.
 * xform: DYMU_XFORM_NONE or DYMU_XFORM_INF_TO_MINUS1. */
int dymu_set_total_cost_export(dymu_ctx* ctx, double* host, size_t ld, int xform, int* direct);
int dymu_download_total_cost_end(dymu_ctx* ctx);
/* values of a plane at n cells (k = j*nx+i), for getTotalCost(Waypoint) G.cpp:860-890 */
int dymu_read_cells(dymu_ctx* ctx, int plane, uint32_t slot, const uint32_t* cell_index,
                    uint32_t n, double* out);

/* All fields of one global node in one round trip (globalNode view, H.hpp:69-108):
 * out[0..9] = elevation, slope, raw_cost, cost, hazard_density, trafficability,
 * total_cost (slot 0), terrain, isObstacle, locomotion mode index (255 = DONT_CARE). */
int dymu_read_node(dymu_ctx* ctx, uint32_t i, uint32_t j, double out[10]);
/* number of cells of a slot with total cost <= threshold (CLOSED-set size) */
int dymu_count_leq(dymu_ctx* ctx, uint32_t slot, double threshold, uint64_t* n);

/* ---- global path extraction ------------------------------------------------------ */
#define DYMU_PATH_OK 0
#define DYMU_PATH_NAN 1        /* first step NaN: G.cpp:628-633 */
#define DYMU_PATH_STALLED 2    /* step < 0.01*tau*res: G.cpp:650-656 */
#define DYMU_PATH_CAPACITY 3   /* output buffer exhausted (reference loop is unbounded) */
#define DYMU_PATH_OUTSIDE 4    /* left the grid (reference would dereference NULL) */
/* computeGlobalPath, G.cpp:615-714: gradient descent on the device-resident total-cost
 * plane.  (x0, y0) offset-free metres.  Each output waypoint is 5 doubles
 * {x, y, z, dCostX, dCostY}: the heading of waypoint k+1 is atan2(-dCostY_k, -dCostX_k)
 * (G.cpp:709), left to the host so that libm's atan2 is the one used. The goal
 * waypoint (G.cpp:659-660) is NOT appended. */
int dymu_extract_global_path(dymu_ctx* ctx, uint32_t slot, double x0, double y0, double tau,
                             uint32_t goal_i, uint32_t goal_j, double* out, uint32_t cap,
                             uint32_t* n_out, int* status);

/* Batched variant: query q descends on slot slots[q] from (xy0[2q], xy0[2q+1]) to goal
 * (goal_ij[2q], goal_ij[2q+1]); one CTA per query, all in one launch.  out holds n*cap*5
 * doubles (query q at out + q*cap*5); n_out / status hold n entries. */
int dymu_extract_global_path_batch(dymu_ctx* ctx, uint32_t n, const uint32_t* slots,
                                   const double* xy0, double tau, const uint32_t* goal_ij,
                                   double* out, uint32_t cap, uint32_t* n_out, int* status);

/* ---- several GPUs behind one call (SURVEY.md section 8e) ------------------------------- */
/* Batches of independent goal queries: context k (its own GPU, its own copy of the cost map,
 * dymu_reserve_slots goals per launch) gets the k-th contiguous block of the n_goals queries; one
 * host thread per context, no data-path exchange.  Per query: computeEntireTotalCostMap
 * (G.cpp:443-468) and, if `paths` is given, the descent from (start_xy[2q], start_xy[2q+1])
 * (G.cpp:615-714) into paths + q*cap*5 (format of dymu_extract_global_path), path_len[q],
 * path_status[q].  ms_per_ctx (optional): host wall time of each context's share. */
int dymu_batch_solve(dymu_ctx** ctxs, uint32_t n_ctx, uint32_t n_goals, const uint32_t* goal_i,
                     const uint32_t* goal_j, const double* start_xy, double tau, double* paths,
                     uint32_t cap, uint32_t* path_len, int32_t* path_status, float* ms_per_ctx);

typedef struct dymu_dd_stats
{
    uint32_t rounds;            /* exchange rounds */
    uint32_t converged;
    float wall_ms;              /* host wall clock of the whole solve */
    float max_kernel_ms;        /* solver kernel time of the busiest strip */
    float sum_kernel_ms;        /* ... summed over the strips */
    uint32_t reserved_;
    uint64_t tile_activations;  /* summed over the strips */
    uint64_t cell_updates;
} dymu_dd_stats;

/* One grid cut into n row strips, strip k on context k: global rows [cuts[k], cuts[k+1]) plus
 * one ghost row per interior side (cost 0 there), i.e. ctxs[k] has cuts[k+1]-cuts[k] (+1) (+1)
 * rows, the common width, and its cost map set (dymu_set_cost_map on the strip's rows; interior
 * cuts on multiples of the 32-cell tile).  The goal is given in grid coordinates.  Every round a
 * strip runs at most phases_per_round solver phases (0 = 32), then boundary rows travel GPU to
 * GPU (cudaMemcpyPeerAsync) into the neighbours' ghost rows; computeEntireTotalCostMap
 * (G.cpp:443-468) of the whole grid, same fixed point as the single-grid solve.  On return each
 * strip's total-cost plane holds its rows (dymu_download_total_cost; row 0 is the ghost row for
 * k > 0). */
int dymu_dd_solve(dymu_ctx** ctxs, uint32_t n, const uint32_t* cuts, uint32_t goal_i, uint32_t goal_j,
                  uint32_t phases_per_round, dymu_dd_stats* stats);

/* ---- local layer --------------------------------------------------------------------- */
/* The local layer (localNode, H.hpp:42-67) is a dense window of wg x wg global
 * nodes, r = (uint)(global_res/local_res) local cells per node edge, anchored at
 * global node (gx0, gy0).  Planes: risk, deviation, local total_cost (fp64),
 * isObstacle, state (u8). */
#define DYMU_LPLANE_RISK 0
#define DYMU_LPLANE_DEVIATION 1
#define DYMU_LPLANE_TOTAL_COST 2
#define DYMU_LPLANE_U8_OBSTACLE 0
#define DYMU_LPLANE_U8_STATE 1
int dymu_local_create(dymu_ctx* ctx, uint32_t wg);
int dymu_local_anchor(dymu_ctx* ctx, int64_t gx0, int64_t gy0);
/* Moves and/or resizes the window to wg x wg global nodes anchored at (gx0, gy0), keeping the
 * persistent local-node fields (isObstacle, risk) of the area both windows cover -- the reference
 * subdivides on demand and never forgets a local node (L.cpp:150-156, G.cpp:36).  Deviation,
 * local total cost and state start over (they are reset per propagation anyway, L.cpp:589-599).
 * Creates the window if there is none. */
int dymu_local_reshape(dymu_ctx* ctx, uint32_t wg, int64_t gx0, int64_t gy0); /* clears the window */
int dymu_local_info(const dymu_ctx* ctx, int64_t* gx0, int64_t* gy0, uint32_t* wg, uint32_t* r);
/* rectangle of the local window in window-local cell coordinates */
int dymu_local_read_rect(dymu_ctx* ctx, int lplane, uint32_t x0, uint32_t y0, uint32_t w,
                         uint32_t h, double* host);
int dymu_local_read_rect_u8(dymu_ctx* ctx, int lplane, uint32_t x0, uint32_t y0, uint32_t w,
                            uint32_t h, uint8_t* host);
/* Obstacle ingestion, L.cpp:233-277 (mask part): for every pixel inside the map, the
 * local cell it falls in (getLocalNode, L.cpp:160-173) becomes an obstacle with risk 1 if
 * pixel != 0 or the parent global node is an obstacle.  Outputs, in pixel raster order,
 * the NEW obstacle cells: new_cells[k] = window-local cell index (y*W + x).  The
 * hazard-density bumps (L.cpp:264-274) and the path-blocking test (L.cpp:441-471)
 * consume that list. */
int dymu_local_ingest(dymu_ctx* ctx, const uint8_t* image, uint32_t w, uint32_t h,
                      uint32_t row_size, uint32_t pixel_size, double res, double rover_x,
                      double rover_y, uint32_t* new_cells, uint32_t cap, uint32_t* n_new);
/* isBlockingObstacle over a list of obstacle cells, L.cpp:441-471: returns the
 * accumulated minIndex / maxIndex and whether any obstacle blocks the path. */
int dymu_local_blocking(dymu_ctx* ctx, const uint32_t* cells, uint32_t n_cells,
                        const double* path_xy, uint32_t n_path, double risk_distance,
                        uint32_t* min_index, uint32_t* max_index, int* blocked);
/* expandRisk, L.cpp:493-576: fixed point of propagateRisk from all obstacle cells. */
int dymu_local_expand_risk(dymu_ctx* ctx, double risk_distance, dymu_solve_stats* stats);
/* computeLocalPropagation, L.cpp:578-805: narrow-band march on `deviation` in the
 * reference's exact pop order (vector position tie-break included).
 * approach: 0 CONSERVATIVE (end node given), 1 SWEEPING (end node discovered).
 * Returns end cell (window-local index) or -1 when the reference returns NULL. */
int dymu_local_propagate(dymu_ctx* ctx, int approach, double start_x, double start_y,
                         double overtake_x, double overtake_y, double t_overtake,
                         double risk_ratio, int64_t* end_cell, uint32_t* status,
                         uint64_t* n_closed);
#define DYMU_LOCAL_OK 0
#define DYMU_LOCAL_START_IN_OBSTACLE 1
#define DYMU_LOCAL_END_IN_OBSTACLE 2
#define DYMU_LOCAL_EXHAUSTED 3      /* narrow band drained (reference: watchdog / crash) */
#define DYMU_LOCAL_WINDOW_EXCEEDED 4 /* the wave reached the window border */
/* getLocalPath, L.cpp:807-1023.  Output waypoints {x, y, z, dCostX, dCostY, kind}:
 * kind 0 = gradient step (heading atan2(dCostY,dCostX), L.cpp:974), 1 = Dijkstra
 * fallback step (heading atan2(dCostY,dCostX) with the stored deltas, L.cpp:866-867),
 * 2 = first waypoint whose gradient step was rejected (heading of the end node, L.cpp:815).
 * (offset_x, offset_y) = global_offset, subtracted once more for the elevation look-up
 * exactly as L.cpp:890-891 does.
 * Stored in the order the reference inserts them (last inserted = front). */
int dymu_local_extract_path(dymu_ctx* ctx, int64_t end_cell, double start_x, double start_y,
                            double offset_x, double offset_y, double* out, uint32_t cap,
                            uint32_t* n_out, int* status);
/* per window global node (wg*wg bytes, row-major): 1 if the last propagation looked into a
 * local node of that global node from a different parent, i.e. the reference would have
 * called subdivideGlobalNode on it (L.cpp:658-663).  clear != 0 resets the flags. */
int dymu_local_read_entered(dymu_ctx* ctx, uint8_t* host, int clear);
/* risk at the local cells containing n waypoints (evaluatePath, L.cpp:1046-1047);
 * cells outside the window report 0. */
int dymu_local_sample_risk(dymu_ctx* ctx, const double* xy, uint32_t n, double* risk_out);
/* world->window mapping of getLocalNode (L.cpp:160-189); -1 if outside the window */
int dymu_local_cell_of(dymu_ctx* ctx, double x, double y, int64_t* cell);

#ifdef __cplusplus
}
#endif
#endif /* DYMU_CUDA_H */
