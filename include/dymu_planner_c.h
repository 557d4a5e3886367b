/*
 * dymu_planner_c.h -- flat C view of PathPlanning_lib::DyMuPathPlanner.
 *
 * The reference has no C ABI: its interface *is* the C++ class declared in
 * src/DyMu.hpp:397-609.  This header flattens the public methods of that
 * class one-to-one so that Python (ctypes), C and cgo-style callers can drive
 * a planner without C++ types.  The implementation file
 * (planning-path_planning_b200/capi/planner_capi.cpp) contains no planner
 * logic; it is compiled twice from the same source:
 *
 *   - against the unmodified reference headers/sources  -> oracle/_ref/libdymu_ref.so
 *   - against this repository's drop-in DyMu.hpp        -> libdymu_b200.so
 *
 * so every parity test issues literally the same call sequence to both.
 * Each entry point cites the reference method it forwards to.
 *
 * Conventions: matrices are row-major [j][i] (NY rows of NX), doubles.
 * Waypoint arrays are packed {x, y, z, heading} per waypoint.
 * Functions returning `int` for a reference `bool` return 1/0; a negative
 * return is a wrapper-level error (bad handle, buffer too small).
 */
#ifndef DYMU_PLANNER_C_H
#define DYMU_PLANNER_C_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dymu_planner dymu_planner;

/* enum repairingAproach, DyMu.hpp:36-40 */
#define DYMU_CONSERVATIVE 0
#define DYMU_SWEEPING 1

/* matrix kinds for dymu_planner_get_matrix */
#define DYMU_MAT_TOTAL_COST 0     /* getTotalCostMatrix      G.cpp:799-811 (inf -> -1) */
#define DYMU_MAT_GLOBAL_COST 1    /* getGlobalCostMatrix     G.cpp:815-829 (obstacle -> -1) */
#define DYMU_MAT_HAZARD_DENSITY 2 /* getHazardDensityMatrix  G.cpp:833-842 */
#define DYMU_MAT_TRAFFICABILITY 3 /* getTrafficabilityMatrix G.cpp:846-855 */

/* local window kinds for dymu_planner_get_local_matrix */
#define DYMU_LOCAL_RISK 0      /* getRiskMatrix      L.cpp:1111-1158 */
#define DYMU_LOCAL_DEVIATION 1 /* getDeviationMatrix L.cpp:1160-1211 */

/* per-node field taps (globalNode members, DyMu.hpp:69-108) */
#define DYMU_NODE_ELEVATION 0
#define DYMU_NODE_SLOPE 1
#define DYMU_NODE_RAW_COST 2
#define DYMU_NODE_COST 3
#define DYMU_NODE_IS_OBSTACLE 4
#define DYMU_NODE_STATE 5 /* 0 OPEN, 1 CLOSED */
#define DYMU_NODE_HAS_LOCAL_MAP 6
#define DYMU_NODE_TERRAIN 7
#define DYMU_NODE_TOTAL_COST_RAW 8 /* total_cost with +inf kept */

/* "reference" or "b200" */
const char* dymu_planner_impl(void);

/* DyMuPathPlanner::DyMuPathPlanner, G.cpp:22-33 */
dymu_planner* dymu_planner_create(double risk_distance, double reconnect_distance,
                                  double risk_ratio, int approach);
/* DyMuPathPlanner::~DyMuPathPlanner, G.cpp:36 */
void dymu_planner_destroy(dymu_planner* p);

/* initGlobalLayer, G.cpp:39-104 */
int dymu_planner_init_global_layer(dymu_planner* p, double global_res, double local_res,
                                   unsigned num_nodes_x, unsigned num_nodes_y, double offset_x,
                                   double offset_y);
/* setCostMap, G.cpp:109-126 */
int dymu_planner_set_cost_map(dymu_planner* p, const double* cost, unsigned ny, unsigned nx);
/* computeCostMap, G.cpp:145-181.  locomotion_modes: comma-separated names. */
int dymu_planner_compute_cost_map(dymu_planner* p, const double* cost_data, int n_cost_data,
                                  const double* slope_values, int n_slopes,
                                  const char* locomotion_modes, const double* elevation,
                                  const double* terrain, unsigned ny, unsigned nx);
/* setGoal, G.cpp:322-357 */
int dymu_planner_set_goal(dymu_planner* p, double x, double y, double heading);
/* computeTotalCostMap, G.cpp:364-408 */
int dymu_planner_compute_total_cost_map(dymu_planner* p, double x, double y);
/* computeEntireTotalCostMap, G.cpp:443-468 */
int dymu_planner_compute_entire_total_cost_map(dymu_planner* p);
/* getPath, G.cpp:589-611.  Returns the number of waypoints of the result
 * (which may exceed `cap`; only min(n, cap) are written). */
int dymu_planner_get_path(dymu_planner* p, double x, double y, double* xyzh, int cap);
/* computeGlobalPath, G.cpp:615-662 (argument already offset-free, as in the reference) */
int dymu_planner_compute_global_path(dymu_planner* p, double x, double y);
/* public member current_path, DyMu.hpp:456 */
int dymu_planner_get_current_path(dymu_planner* p, double* xyzh, int cap);
/* matrix getters, G.cpp:799-855.  `out` holds NY*NX doubles. */
int dymu_planner_get_matrix(dymu_planner* p, int kind, double* out);
/* getTotalCost(Waypoint), G.cpp:860-890 */
double dymu_planner_get_total_cost(dymu_planner* p, double x, double y);
/* getLocomotionMode, G.cpp:788-795 */
int dymu_planner_get_locomotion_mode(dymu_planner* p, double x, double y, char* buf, int cap);
/* computeLocalPlanning, L.cpp:193-291.  `image` is h rows of w uint8 pixels
 * (row_size = w, pixel_size = 1).  *n_traj receives trajectory.size(). */
int dymu_planner_compute_local_planning(dymu_planner* p, double x, double y,
                                        const uint8_t* image, int w, int h, double res,
                                        double* traj_xyzh, int cap, int* n_traj,
                                        double* local_time_s);
/* getRiskMatrix / getDeviationMatrix, L.cpp:1111-1211.  Returns the side
 * length S of the square window; writes S*S doubles if S*S <= cap. */
int dymu_planner_get_local_matrix(dymu_planner* p, int kind, double x, double y, double* out,
                                  int cap);
/* getReconnectingIndex, L.cpp:1213 */
int dymu_planner_get_reconnecting_index(dymu_planner* p);
/* public member remaining_total_cost, DyMu.hpp:464 */
double dymu_planner_get_remaining_total_cost(dymu_planner* p);
/* Per-node taps through getGlobalNode(i,j) (G.cpp:313-317); `out` holds
 * NY*NX doubles (booleans/enums as 0/1). */
int dymu_planner_get_node_field(dymu_planner* p, int field, double* out);
/* ---- CoRa: cost ratio updating after traverse, G.cpp:895-1038 ---- */
/* initCoRaMethod, G.cpp:895-922 */
int dymu_planner_cora_init(dymu_planner* p, int num_terrains, int num_criteria, const double* weights,
                           int n_weights);
/* getTerrain, G.cpp:941-950 (position in world coordinates) */
int dymu_planner_get_terrain(dymu_planner* p, double x, double y);
/* fillTerrainInfo, G.cpp:926-938 */
int dymu_planner_fill_terrain_info(dymu_planner* p, int terrain_id, const double* data, int n);
/* updateCost, G.cpp:956-993.  Returns the table length; writes min(len, cap) entries. */
int dymu_planner_update_cost(dymu_planner* p, double* lut, int cap);
/* computeCostRatio, G.cpp:999-1038.  Returns the number of ratios. */
int dymu_planner_compute_cost_ratio(dymu_planner* p, double* ratios, int cap);
/* Re-run computeCostMap (G.cpp:145-181) with the planner's current public cost_lutable and
 * the slope values / locomotion modes / maps of the last dymu_planner_compute_cost_map call:
 * the step a CoRa caller performs after updateCost.  The reference build re-sends the maps it
 * kept on the host; the B200 build rebuilds from the planes resident in HBM
 * (DyMuPathPlanner::recomputeCostMap). */
int dymu_planner_recompute_cost_map(dymu_planner* p);

/* seconds spent inside the last call of the given kind (wrapper-side
 * steady_clock around the forwarded method; conversions excluded) */
/* Node-level steps of the reference class (H.hpp:520-536), on node (i, j) / waypoint (x, y):
 * gradientNode G.cpp:718-772; computeNextGlobalWaypoint G.cpp:666-714 (out = next x, next y,
 * heading, interpolated z of the input waypoint); propagateGlobalNode G.cpp:500-546 (returns the
 * node's total cost after the update).  Return 0 when the node does not exist. */
int dymu_planner_gradient_node(dymu_planner* p, unsigned i, unsigned j, double* dnx, double* dny);
int dymu_planner_next_global_waypoint(dymu_planner* p, double x, double y, double tau, double out[4]);
int dymu_planner_propagate_global_node(dymu_planner* p, unsigned i, unsigned j, double* total_cost);

/* Copy-free variants (extensions of the B200 drop-in; the reference build implements them on top
 * of the by-value methods so that the same call sequence runs on both):
 *   set_cost_map_flat          setCostMap(const double*, ld) -- with a goal in place the upload is
 *                              streamed behind the next computeEntireTotalCostMap; the buffer must
 *                              stay unchanged until that call returns
 *   set_total_cost_target      setTotalCostMatrixTarget(out, ld): deliver the total-cost matrix
 *                              into `out` right after every solve
 *   get_total_cost_matrix_flat getTotalCostMatrix(out, ld) */
int dymu_planner_set_cost_map_flat(dymu_planner* p, const double* cost, unsigned ld);
int dymu_planner_set_total_cost_target(dymu_planner* p, double* out, unsigned ld);
int dymu_planner_get_total_cost_matrix_flat(dymu_planner* p, double* out, unsigned ld);
/* setSlopeAnisotropy(angles, factors) (extension of the B200 drop-in): n pairs of signed slope
 * angle in degrees and cost factor, n = 0 switches it off; 1 = applied, 0 = rejected.  The
 * reference has no such capability: its build returns -1. */
int dymu_planner_set_slope_anisotropy(dymu_planner* p, const double* angles, const double* factors, int n);
/* setObstacleClearance(radius, margin, penalty) (extension of the B200 drop-in, metres): lethal
 * radius and penalised margin around obstacle nodes, radius = margin = 0 switches it off; 1 = applied,
 * 0 = rejected.  The reference has no such capability: its build returns -1. */
int dymu_planner_set_obstacle_clearance(dymu_planner* p, double radius, double margin, double penalty);

double dymu_planner_last_call_seconds(dymu_planner* p);

#ifdef __cplusplus
}
#endif
#endif /* DYMU_PLANNER_C_H */
