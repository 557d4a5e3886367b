// DyMuGlobalLayer.cpp -- host side of the drop-in DyMuPathPlanner, global layer.
//
// Mirrors the public behaviour of the reference's src/DyMu_GlobalPathPlanning.cpp
// ("G.cpp"): same argument meaning, same bool / NULL error convention, same coordinate
// handling (global_offset subtracted on entry, re-added by getPath).  All per-node work is
// delegated to the CUDA C ABI (include/dymu_cuda.h); what stays here is the scalar
// validation logic around the goal and the start node and the assembly of waypoints.
#include "DyMu.hpp"

#include <algorithm>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include "dymu_cuda.h"
#include "DyMuTiming.hpp"
#include "dymu_planner_c.h"

using namespace PathPlanning_lib;

namespace
{
const double kInf = std::numeric_limits<double>::infinity();
}

/*****************************CONSTRUCTOR**************************************/
// reference: G.cpp:22-33
DyMuPathPlanner::DyMuPathPlanner(double risk_distance,
                                 double reconnect_distance,
                                 double risk_ratio,
                                 repairingAproach input_approach)
    : dev(NULL),
      num_nodes_X(0),
      num_nodes_Y(0),
      global_res(1.0),
      local_res(1.0),
      res_ratio(1),
      risk_distance(risk_distance),
      reconnect_distance(reconnect_distance),
      risk_ratio(risk_ratio),
      repairing_approach(input_approach),
      num_terrains(0),
      num_criteria(0),
      base_speed(0.0),
      goal_set(false),
      goal_i(0),
      goal_j(0),
      closed_threshold(kInf),
      readback_target(NULL),
      readback_ld(0),
      readback_inflight(false),
      streamed_cost(false),
      clearance_radius(0.0),
      pending_risk(false),
      local_window_nodes(64),
      local_ready(false),
      local_created(false),
      local_agent_cell(-1)
{
    global_goal = NULL;
    local_agent = NULL;
    remaining_total_cost = 0.0;
    reconnecting_index = 0;
    if (const char* e = getenv("DYMU_LOCAL_WG"))
        if (atoi(e) >= 8) local_window_nodes = (uint)atoi(e);
}

/******************************DESTRUCTOR**************************************/
// The reference leaks every node (G.cpp:36); the device planes are released here.
DyMuPathPlanner::~DyMuPathPlanner()
{
    finishReadback();
    if (dev) dymu_destroy(dev);
    dev = NULL;
}

bool DyMuPathPlanner::deviceOk(int rc, const char* what)
{
    if (rc == DYMU_OK) return true;
    last_error = std::string(what) + ": " + (dev ? dymu_last_error(dev) : "no device context");
    LOG_ERROR_S << "PLANNER (B200): " << last_error;
    if (getenv("DYMU_VERBOSE")) fprintf(stderr, "dymu_b200: %s (rc=%d)\n", last_error.c_str(), rc);
    return false;
}

/*******************GLOBAL_LAYER_INITIALIZATION********************************/
// reference: G.cpp:39-104.  Allocation of the SoA planes replaces the per-node `new`
// and the neighbour wiring (neighbours are index arithmetic on the device).
bool DyMuPathPlanner::initGlobalLayer(double globalres,
                                      double localres,
                                      uint numnodesX,
                                      uint numnodesY,
                                      std::vector<double> offset)
{
    global_res = globalres;
    local_res = localres;
    num_nodes_X = numnodesX;
    num_nodes_Y = numnodesY;
    res_ratio = (uint)(global_res / local_res);
    global_offset = offset;
    if (global_offset.size() < 2) global_offset.resize(2, 0.0);
    finishReadback();
    if (dev)
    {
        dymu_destroy(dev);
        dev = NULL;
    }
    int rc = dymu_create(-1, num_nodes_X, num_nodes_Y, global_res, local_res, &dev);
    if (rc != DYMU_OK)
    {
        deviceOk(rc, "initGlobalLayer");
        if (dev) dymu_destroy(dev);
        dev = NULL;
        return false;
    }
    has_local.assign((size_t)num_nodes_X * num_nodes_Y, 0);
    global_views.clear();
    local_views.clear();
    goal_set = false;
    global_goal = NULL;
    closed_threshold = kInf;
    clearance_radius = 0.0;
    pending_risk = false;
    local_ready = false;
    // the local window is allocated up front (the reference builds its whole node graph here): the
    // first repair does not pay for cudaMalloc
    local_created = deviceOk(dymu_local_create(dev, local_window_nodes), "local window");
    if (readback_target && readback_ld >= num_nodes_X)
    {
        int direct = 0;  // the matrix target outlives a re-initialisation
        dymu_set_total_cost_export(dev, readback_target, readback_ld, DYMU_XFORM_INF_TO_MINUS1, &direct);
    }
    return true;
}

/*******************USING PREVIOUSLY DEFINED COST MAP**************************/
// reference: G.cpp:109-126
bool DyMuPathPlanner::setCostMap(std::vector<std::vector<double>> cost_map)
{
    if (!dev) return false;
    if ((cost_map.size() != num_nodes_Y) || (cost_map[0].size() != num_nodes_X)) return false;
    std::vector<double> flat((size_t)num_nodes_X * num_nodes_Y);
    for (uint j = 0; j < num_nodes_Y; j++)
    {
        if (cost_map[j].size() != num_nodes_X) return false;
        std::copy(cost_map[j].begin(), cost_map[j].end(), flat.begin() + (size_t)j * num_nodes_X);
    }
    // `flat` dies with this call: blocking upload
    return deviceOk(dymu_set_cost_map(dev, flat.data(), num_nodes_X), "setCostMap");
}

// Flat variant.  With a goal in place the upload is streamed: the rows around the goal go first
// and the call returns without waiting; computeEntireTotalCostMap() starts on those rows while the
// rest arrives (dymu_set_cost_map_begin).  The buffer must stay unchanged until the next planner
// call returns.  Every other planner call completes the upload first, so the observable state is
// the reference's.
bool DyMuPathPlanner::setCostMap(const double* cost_map, size_t ld)
{
    if (!dev || !cost_map) return false;
    finishReadback();
    if (goal_set)
    {
        streamed_cost = deviceOk(dymu_set_cost_map_begin(dev, cost_map, ld, goal_j), "setCostMap");
        return streamed_cost;
    }
    return deviceOk(dymu_set_cost_map(dev, cost_map, ld), "setCostMap");
}

bool DyMuPathPlanner::setSlopeAnisotropy(const std::vector<double>& slope_angles_deg,
                                         const std::vector<double>& factors)
{
    if (!dev || slope_angles_deg.size() != factors.size() || slope_angles_deg.size() > DYMU_ANISO_MAX) return false;
    finishReadback();
    return deviceOk(dymu_set_anisotropy(dev, slope_angles_deg.data(), factors.data(), (int)factors.size()),
                    "setSlopeAnisotropy");
}

bool DyMuPathPlanner::setObstacleClearance(double radius, double margin, double penalty)
{
    if (!dev) return false;
    finishReadback();
    if (!deviceOk(dymu_set_obstacle_clearance(dev, radius, margin, penalty), "setObstacleClearance")) return false;
    clearance_radius = (radius == 0 && margin == 0) ? 0.0 : radius;
    return true;
}

// The obstacle-goal rule extended to the lethal ring of the obstacle clearance: the rover cannot stand
// on a goal whose clearance is <= radius, so it is refused like a goal on an obstacle.
bool DyMuPathPlanner::goalInLethalRing()
{
    if (!(clearance_radius > 0)) return false;
    uint32_t idx = goal_j * num_nodes_X + goal_i;
    double d = kInf;
    if (!deviceOk(dymu_read_cells(dev, DYMU_PLANE_CLEARANCE, 0, &idx, 1, &d), "goal clearance")) return true;
    return d <= clearance_radius;
}

void DyMuPathPlanner::finishReadback()
{
    if (readback_inflight && dev) deviceOk(dymu_download_total_cost_end(dev), "getTotalCostMatrix");
    readback_inflight = false;
}

// Total-cost matrix delivery (extension): after every successful compute*TotalCostMap the matrix
// (inf -> -1, G.cpp:799-811) is copied into `out` on the copy stream, overlapping whatever the
// caller does next (getPath); getTotalCostMatrix(out, ld) with the same pointer then only waits for
// that copy.  NULL switches it off.
// When `out` is page-locked memory the device can write to (cudaHostAlloc / cudaHostRegister, a torch
// pinned tensor), a solve from scratch stores the matrix there itself while it runs -- every tile as
// soon as the wave front is past it (dymu_set_total_cost_export) -- and there is no copy left to wait
// for.  `out` must stay valid until the target is changed or switched off.
void DyMuPathPlanner::setTotalCostMatrixTarget(double* out, size_t ld)
{
    finishReadback();
    readback_target = out;
    readback_ld = ld;
    if (dev)
    {
        int direct = 0;
        deviceOk(dymu_set_total_cost_export(dev, out, ld, DYMU_XFORM_INF_TO_MINUS1, &direct),
                 "setTotalCostMatrixTarget");
    }
}

void DyMuPathPlanner::startReadback()
{
    if (!readback_target || !dev) return;
    readback_inflight = deviceOk(dymu_download_total_cost_begin(dev, 0, readback_target, readback_ld,
                                                                DYMU_XFORM_INF_TO_MINUS1),
                                 "getTotalCostMatrix");
}

/*******************COMPUTE COST MAP FROM SLOPE MAP****************************/
// reference: G.cpp:145-181 (+ calculateSlope 186-210, calculateNominalCost 217-293,
// smoothCost 297-308, all on the device)
bool DyMuPathPlanner::computeCostMap(std::vector<double> cost_data,
                                     std::vector<double> slope_values,
                                     std::vector<std::string> locomotionModes,
                                     std::vector<std::vector<double>> elevation,
                                     std::vector<std::vector<double>> terrainMap)
{
    if (!dev)
    {
        // like the reference (G.cpp:151-153) the tables are recorded before anything can fail
        this->cost_lutable = cost_data;
        this->slope_range = slope_values;
        this->locomotion_modes = locomotionModes;
        return false;
    }
    if (elevation.size() != num_nodes_Y || terrainMap.size() != num_nodes_Y) return false;
    size_t n = (size_t)num_nodes_X * num_nodes_Y;
    std::vector<double> e(n), t(n);
    for (uint j = 0; j < num_nodes_Y; j++)
    {
        if (elevation[j].size() != num_nodes_X || terrainMap[j].size() != num_nodes_X) return false;
        std::copy(elevation[j].begin(), elevation[j].end(), e.begin() + (size_t)j * num_nodes_X);
        std::copy(terrainMap[j].begin(), terrainMap[j].end(), t.begin() + (size_t)j * num_nodes_X);
    }
    return computeCostMap(cost_data, slope_values, locomotionModes, e.data(), num_nodes_X, t.data(),
                          num_nodes_X);
}

bool DyMuPathPlanner::computeCostMap(const std::vector<double>& cost_data,
                                     const std::vector<double>& slope_values,
                                     const std::vector<std::string>& locomotionModes,
                                     const double* elevation, size_t ld_e,
                                     const double* terrainMap, size_t ld_t)
{
    // recorded first, like the reference (G.cpp:151-153), also when the call then fails
    this->cost_lutable = cost_data;
    this->slope_range = slope_values;
    this->locomotion_modes = locomotionModes;
    if (!dev) return false;
    if (cost_data.empty() || slope_values.empty() || locomotionModes.empty()) return false;
    // The reference indexes the table with terrain*range*numLocs + ... without any bound
    // check (G.cpp:237-286); refuse maps whose terrain ids do not fit the table.
    size_t per_terrain = slope_values.size() * locomotionModes.size();
    if (terrainMap)
    {
        double tmax = 0;
        for (uint j = 1; j + 1 < num_nodes_Y; j++)
            for (uint i = 1; i + 1 < num_nodes_X; i++)
                tmax = std::max(tmax, terrainMap[(size_t)j * ld_t + i]);
        if (((size_t)tmax + 1) * per_terrain > cost_data.size())
        {
            last_error = "computeCostMap: cost table too small for the terrain ids in terrainMap";
            LOG_ERROR_S << last_error;
            return false;
        }
    }
    return deviceOk(dymu_compute_cost_map(dev, cost_data.data(), (int)cost_data.size(),
                                          slope_values.data(), (int)slope_values.size(),
                                          (int)locomotionModes.size(), elevation, ld_e, terrainMap,
                                          ld_t),
                    "computeCostMap");
}

/*****************************GET GLOBAL NODE**********************************/
// reference: G.cpp:313-317.  Returns a value view refreshed from the device.
bool DyMuPathPlanner::readNode(uint i, uint j, globalNode& out)
{
    double f[10];
    if (!dev || !deviceOk(dymu_read_node(dev, i, j, f), "getGlobalNode")) return false;
    out.pose.position[0] = (double)i;
    out.pose.position[1] = (double)j;
    out.world_pose.position[0] = (double)i * global_res;
    out.world_pose.position[1] = (double)j * global_res;
    out.elevation = f[0];
    out.slope = f[1];
    out.raw_cost = f[2];
    out.cost = f[3];
    out.hazard_density = f[4];
    out.trafficability = f[5];
    out.total_cost = f[6];
    out.terrain = (unsigned int)f[7];
    out.isObstacle = f[8] != 0.0;
    int lm = (int)f[9];
    out.nodeLocMode = (lm >= 0 && lm < (int)locomotion_modes.size()) ? locomotion_modes[lm]
                                                                     : std::string("DONT_CARE");
    out.state = (f[6] < kInf && f[6] <= closed_threshold) ? CLOSED : OPEN;
    out.hasLocalMap = has_local[(size_t)j * num_nodes_X + i] != 0;
    return true;
}

globalNode* DyMuPathPlanner::getGlobalNode(uint i, uint j)
{
    if ((i >= num_nodes_X) || (j >= num_nodes_Y)) return NULL;
    unsigned long long key = (unsigned long long)j * num_nodes_X + i;
    globalNode& v = global_views[key];
    if (!readNode(i, j, v)) return NULL;
    return &v;
}

long DyMuPathPlanner::nearestIndex(double x, double y) const
{
    // getNearestGlobalNode, G.cpp:572-584 (a negative coordinate wraps to a huge uint -> NULL)
    double fx = x / global_res + 0.5, fy = y / global_res + 0.5;
    if (!(fx >= 0.0) || !(fy >= 0.0) || !(fx < 4294967296.0) || !(fy < 4294967296.0)) return -1;
    uint i = (uint)fx, j = (uint)fy;
    if (i >= num_nodes_X || j >= num_nodes_Y) return -1;
    return (long)j * num_nodes_X + i;
}

/**************************PLACING THE GOAL************************************/
// reference: G.cpp:322-357
bool DyMuPathPlanner::setGoal(base::Waypoint wGoal)
{
    if (!dev) return false;
    wGoal.position[0] = (wGoal.position[0] - global_offset[0]) / global_res;
    wGoal.position[1] = (wGoal.position[1] - global_offset[1]) / global_res;
    if ((wGoal.position[0] < 0) || (wGoal.position[1] < 0)) return false;
    if (!(wGoal.position[0] + 0.5 < 4294967296.0) || !(wGoal.position[1] + 0.5 < 4294967296.0))
        return false;
    uint scaledX = (uint)(wGoal.position[0] + 0.5);
    uint scaledY = (uint)(wGoal.position[1] + 0.5);
    // out of boundaries or on the border (a NULL 4-neighbour)
    if (scaledX >= num_nodes_X || scaledY >= num_nodes_Y) return false;
    if (scaledX == 0 || scaledY == 0 || scaledX + 1 >= num_nodes_X || scaledY + 1 >= num_nodes_Y)
        return false;
    // not next to an obstacle global node
    unsigned char ob[9];
    if (!deviceOk(dymu_read_rect_u8(dev, DYMU_PLANE_U8_OBSTACLE, scaledX - 1, scaledY - 1, 3, 3, ob),
                  "setGoal"))
        return false;
    if (ob[4] || ob[1] || ob[3] || ob[5] || ob[7]) return false;
    goal_set = true;
    goal_i = scaledX;
    goal_j = scaledY;
    readNode(goal_i, goal_j, goal_view);
    goal_view.pose.orientation = wGoal.heading;
    global_goal = &goal_view;
    return true;
}

/***********************COMPUTATION OF TOTAL COST******************************/
// reference: G.cpp:364-408.  The device computes the converged map; the reference's early
// stop (start node and its 4 neighbours CLOSED) is reproduced as the threshold
// T_stop = max of those five values: nodes with total_cost <= T_stop are exactly the ones
// the reference has CLOSED at that moment, and they hold identical (final) values.  Nodes
// beyond T_stop keep their converged values here, whereas the reference leaves tentative
// narrow-band values / infinity there (DESIGN.md, "early stop").
bool DyMuPathPlanner::computeTotalCostMap(base::Waypoint wPos)
{
    if (!dev) return false;
    finishReadback();
    wPos.position[0] -= global_offset[0];
    wPos.position[1] -= global_offset[1];

    if ((global_goal == NULL) || !goal_set)
    {
        LOG_WARN_S << "The goal is not valid";
        return false;
    }
    readNode(goal_i, goal_j, goal_view);
    if (goal_view.isObstacle || goalInLethalRing())
    {
        LOG_WARN_S << "The goal is not valid";
        return false;
    }
    long s = nearestIndex(wPos.position[0], wPos.position[1]);
    if (s < 0) return false;  // the reference dereferences NULL here
    uint si = (uint)(s % num_nodes_X), sj = (uint)(s / num_nodes_X);
    // isSafeNode, G.cpp:410-422 (needs the full 8-neighbourhood)
    if (si == 0 || sj == 0 || si + 1 >= num_nodes_X || sj + 1 >= num_nodes_Y) return false;
    unsigned char ob[9];
    if (!deviceOk(dymu_read_rect_u8(dev, DYMU_PLANE_U8_OBSTACLE, si - 1, sj - 1, 3, 3, ob),
                  "computeTotalCostMap"))
        return false;
    for (int k = 0; k < 9; ++k)
        if (ob[k])
        {
            LOG_ERROR_S << "PLANNER: The rover is located too close to an obstacle";
            return false;
        }
    uint32_t gi = goal_i, gj = goal_j;
    dymu_solve_stats st;
    if (!deviceOk(dymu_solve_incremental(dev, gi, gj, &st, NULL), "computeTotalCostMap")) return false;
    double t_stop = kInf;
    if (!deviceOk(dymu_stop_threshold(dev, 0, si, sj, &t_stop), "computeTotalCostMap")) return false;
    closed_threshold = t_stop;
    readNode(goal_i, goal_j, goal_view);
    goal_view.pose.orientation = global_goal->pose.orientation;
    if (!(t_stop < kInf))
    {
        // the wave cannot close the start neighbourhood: the narrow band drains (G.cpp:399-403)
        LOG_ERROR_S << "The goal is unreachable";
        return false;
    }
    // The reference also answers "unreachable" when the narrow band happens to be empty at
    // the moment the start neighbourhood closes, i.e. nothing reachable lies beyond T_stop.
    uint64_t reached = 0, closed = 0;
    if (deviceOk(dymu_count_reached(dev, 0, &reached), "computeTotalCostMap")
        && deviceOk(dymu_count_leq(dev, 0, t_stop, &closed), "computeTotalCostMap")
        && reached == closed)
    {
        LOG_ERROR_S << "The goal is unreachable";
        return false;
    }
    startReadback();
    return true;
}

// reference: G.cpp:410-422
bool DyMuPathPlanner::isSafeNode(globalNode* global_node)
{
    if (!global_node || !dev) return false;
    uint i = (uint)global_node->pose.position[0], j = (uint)global_node->pose.position[1];
    if (i == 0 || j == 0 || i + 1 >= num_nodes_X || j + 1 >= num_nodes_Y) return false;
    unsigned char ob[9];
    if (!deviceOk(dymu_read_rect_u8(dev, DYMU_PLANE_U8_OBSTACLE, i - 1, j - 1, 3, 3, ob), "isSafeNode"))
        return false;
    for (int k = 0; k < 9; ++k)
        if (ob[k]) return false;
    return true;
}

// reference: G.cpp:424-436 (CLOSED == total_cost <= closed_threshold)
bool DyMuPathPlanner::isFullyClosedNode(globalNode* global_node)
{
    if (!global_node || !dev) return false;
    uint i = (uint)global_node->pose.position[0], j = (uint)global_node->pose.position[1];
    if (i == 0 || j == 0 || i + 1 >= num_nodes_X || j + 1 >= num_nodes_Y) return false;
    uint32_t idx[5] = {j * num_nodes_X + i, (j - 1) * num_nodes_X + i, j * num_nodes_X + i - 1,
                       j * num_nodes_X + i + 1, (j + 1) * num_nodes_X + i};
    double v[5];
    if (!deviceOk(dymu_read_cells(dev, DYMU_PLANE_TOTAL_COST, 0, idx, 5, v), "isFullyClosedNode"))
        return false;
    for (int k = 0; k < 5; ++k)
        if (!(v[k] < kInf && v[k] <= closed_threshold)) return false;
    return true;
}

/***********************COMPUTATION OF TOTAL COST******************************/
// reference: G.cpp:443-468
bool DyMuPathPlanner::computeEntireTotalCostMap()
{
    if (!dev) return false;
    if ((global_goal == NULL) || !goal_set)
    {
        LOG_WARN_S << "The goal is not valid";
        return false;
    }
    finishReadback();
    if (!streamed_cost)
    {
        readNode(goal_i, goal_j, goal_view);
        if (goal_view.isObstacle)
        {
            LOG_WARN_S << "The goal is not valid";
            return false;
        }
    }
    if (goalInLethalRing())
    {
        LOG_WARN_S << "The goal is not valid";
        return false;
    }
    // With a cost map that is still being uploaded (setCostMap(const double*, ld)) the test
    // "global_goal->isObstacle" (G.cpp:447) is left to the solve itself, which starts on the rows
    // that have arrived: a goal on an obstacle cell is not seeded and reported in the statistics.
    // (In that one case the previous total-cost map is already reset when false is returned.)
    uint32_t gi = goal_i, gj = goal_j;
    dymu_solve_stats st;
    // A resident map of the same goal is re-solved incrementally: only what the changes of cost,
    // hazard_density and trafficability since then can have touched (the local layer's feedback,
    // L.cpp:264-274 and 388-394) is propagated again; anything else is a full solve.
    int rc = streamed_cost ? dymu_solve_total_cost(dev, 1, &gi, &gj, &st)
                           : dymu_solve_incremental(dev, gi, gj, &st, NULL);
    streamed_cost = false;
    if (!deviceOk(rc, "computeEntireTotalCostMap")) return false;
    if (st.goal_obstacle)
    {
        LOG_WARN_S << "The goal is not valid";
        return false;
    }
    closed_threshold = kInf;
    double heading = global_goal->pose.orientation;
    readNode(goal_i, goal_j, goal_view);
    goal_view.pose.orientation = heading;
    startReadback();
    return true;
}

// reference: G.cpp:473-496.  The device solve resets the plane itself; kept for API parity.
void DyMuPathPlanner::resetTotalCostMap() { closed_threshold = kInf; }
void DyMuPathPlanner::resetGlobalNarrowBand() {}

/***************************GET NEAREST NODE***********************************/
// reference: G.cpp:572-584
globalNode* DyMuPathPlanner::getNearestGlobalNode(base::Pose2D pos)
{
    long g = nearestIndex(pos.position[0], pos.position[1]);
    if (g < 0) return NULL;
    return getGlobalNode((uint)(g % num_nodes_X), (uint)(g / num_nodes_X));
}

globalNode* DyMuPathPlanner::getNearestGlobalNode(base::Waypoint wPos)
{
    long g = nearestIndex(wPos.position[0], wPos.position[1]);
    if (g < 0) return NULL;
    return getGlobalNode((uint)(g % num_nodes_X), (uint)(g / num_nodes_X));
}

/****************************GET THE PATH**************************************/
// reference: G.cpp:589-611
std::vector<base::Waypoint> DyMuPathPlanner::getPath(base::Waypoint wPos)
{
    wPos.position[0] -= global_offset[0];
    wPos.position[1] -= global_offset[1];
    {
        Lap lap("getPath: computeGlobalPath");
        computeGlobalPath(wPos);
    }
    {
        Lap lap("getPath: evaluatePath");
        evaluatePath(0);
    }
    Lap lap("getPath: copy out");
    std::vector<base::Waypoint> output_path = current_path;
    for (size_t i = 0; i < output_path.size(); i++)
    {
        output_path[i].position[0] += global_offset[0];
        output_path[i].position[1] += global_offset[1];
    }
    return output_path;
}

/*********************COMPUTE GLOBAL PATH**************************************/
// reference: G.cpp:615-662.  The descent runs in a single-warp kernel on the resident
// total-cost plane; it returns positions, the interpolated z and the gradient used at each
// waypoint.  Headings are formed here with the host libm: waypoint k+1 carries
// atan2(-dCostY_k, -dCostX_k) (G.cpp:709), waypoint 0 keeps the caller's heading.
bool DyMuPathPlanner::computeGlobalPath(base::Waypoint wPos)
{
    current_path.clear();
    if (!dev || !goal_set) return false;
    base::Waypoint sinkPoint;
    sinkPoint.position[0] = global_res * (double)goal_i;
    sinkPoint.position[1] = global_res * (double)goal_j;
    sinkPoint.heading = global_goal ? global_goal->pose.orientation : 0.0;

    double tau = std::min(0.4, risk_distance);
    uint32_t cap = 1u << 16, n = 0;
    int status = 0;
    std::vector<double> buf;
    Lap lap_x("  extract + convert");
    for (;;)
    {
        buf.resize((size_t)cap * 5);
        if (!deviceOk(dymu_extract_global_path(dev, 0, wPos.position[0], wPos.position[1], tau, goal_i,
                                               goal_j, buf.data(), cap, &n, &status),
                      "computeGlobalPath"))
            return false;
        if (status != DYMU_PATH_CAPACITY || cap >= (1u << 24)) break;
        cap *= 4;  // the reference loop is unbounded (quirk 8); grow and retry
    }
    if (status == DYMU_PATH_NAN || (status == DYMU_PATH_OUTSIDE && n == 0))
    {
        LOG_ERROR_S << "PLANNER: Gradient Descent Method failed";
        return false;
    }
    current_path.reserve(n + 1);
    for (uint32_t k = 0; k < n; ++k)
    {
        base::Waypoint w;
        w.position[0] = buf[5 * k + 0];
        w.position[1] = buf[5 * k + 1];
        w.position[2] = buf[5 * k + 2];
        if (k == 0) w.heading = wPos.heading;
        else w.heading = atan2(-buf[5 * (k - 1) + 4], -buf[5 * (k - 1) + 3]);
        current_path.push_back(w);
    }
    if (status != DYMU_PATH_OK)
    {
        LOG_ERROR_S << "ERROR in trajectory";
        return false;
    }
    // the goal's elevation is read after the descent: a small device-to-host copy queues behind a
    // total-cost matrix delivery that may be in flight (setTotalCostMatrixTarget), and by now that
    // copy has had the whole descent to finish
    globalNode g;
    readNode(goal_i, goal_j, g);
    sinkPoint.position[2] = g.elevation;
    current_path.push_back(sinkPoint);
    return true;
}

/*************************INTERPOLATION FUNCTION*******************************/
// reference: G.cpp:776-784
double DyMuPathPlanner::interpolate(double a, double b, double g00, double g01, double g10, double g11)
{
    return g00 + (g10 - g00) * a + (g01 - g00) * b + (g11 + g00 - g10 - g01) * a * b;
}

/*************************GET LOCOMOTION MODE**********************************/
// reference: G.cpp:788-795
std::string DyMuPathPlanner::getLocomotionMode(base::Waypoint wPos)
{
    wPos.position[0] -= global_offset[0];
    wPos.position[1] -= global_offset[1];
    globalNode* gNode = getNearestGlobalNode(wPos);
    if (!gNode) return std::string("DONT_CARE");
    return gNode->nodeLocMode;
}

/***********************MATRIX GETTERS******************************************/
namespace
{
std::vector<std::vector<double>> nested(const std::vector<double>& flat, uint ny, uint nx)
{
    std::vector<std::vector<double>> m(ny);
    for (uint j = 0; j < ny; j++)
        m[j].assign(flat.begin() + (size_t)j * nx, flat.begin() + (size_t)(j + 1) * nx);
    return m;
}
}  // namespace

// reference: G.cpp:799-811 (inf -> -1 applied by the read-back kernel)
std::vector<std::vector<double>> DyMuPathPlanner::getTotalCostMatrix()
{
    std::vector<double> flat((size_t)num_nodes_X * num_nodes_Y, -1.0);
    if (dev) deviceOk(dymu_download_total_cost(dev, 0, flat.data(), num_nodes_X, DYMU_XFORM_INF_TO_MINUS1),
                      "getTotalCostMatrix");
    return nested(flat, num_nodes_Y, num_nodes_X);
}

bool DyMuPathPlanner::getTotalCostMatrix(double* out, size_t ld)
{
    if (!dev || !out) return false;
    if (readback_inflight && out == readback_target && ld == readback_ld)
    {
        // already on its way since the solve finished (setTotalCostMatrixTarget)
        bool ok = deviceOk(dymu_download_total_cost_end(dev), "getTotalCostMatrix");
        readback_inflight = false;
        return ok;
    }
    finishReadback();
    return deviceOk(dymu_download_total_cost(dev, 0, out, ld, DYMU_XFORM_INF_TO_MINUS1), "getTotalCostMatrix");
}

// reference: G.cpp:815-829
std::vector<std::vector<double>> DyMuPathPlanner::getGlobalCostMatrix()
{
    std::vector<double> flat((size_t)num_nodes_X * num_nodes_Y, -1.0);
    if (dev) deviceOk(dymu_download_plane(dev, DYMU_PLANE_COST, flat.data(), num_nodes_X,
                                          DYMU_XFORM_EFFECTIVE_COST),
                      "getGlobalCostMatrix");
    return nested(flat, num_nodes_Y, num_nodes_X);
}

// reference: G.cpp:833-842
std::vector<std::vector<double>> DyMuPathPlanner::getHazardDensityMatrix()
{
    std::vector<double> flat((size_t)num_nodes_X * num_nodes_Y, 0.0);
    if (dev) deviceOk(dymu_download_plane(dev, DYMU_PLANE_HAZARD_DENSITY, flat.data(), num_nodes_X,
                                          DYMU_XFORM_NONE),
                      "getHazardDensityMatrix");
    return nested(flat, num_nodes_Y, num_nodes_X);
}

// reference: G.cpp:846-855
std::vector<std::vector<double>> DyMuPathPlanner::getTrafficabilityMatrix()
{
    std::vector<double> flat((size_t)num_nodes_X * num_nodes_Y, 1.0);
    if (dev) deviceOk(dymu_download_plane(dev, DYMU_PLANE_TRAFFICABILITY, flat.data(), num_nodes_X,
                                          DYMU_XFORM_NONE),
                      "getTrafficabilityMatrix");
    return nested(flat, num_nodes_Y, num_nodes_X);
}

/*******************GET THE TOTAL COST OF A LOCATION***************************/
// reference: G.cpp:860-890 on an offset-free position
double DyMuPathPlanner::totalCostNoOffset(double x, double y)
{
    double fx = x / global_res, fy = y / global_res;
    if (!dev || !(fx >= 0) || !(fy >= 0) || !(fx < (double)num_nodes_X) || !(fy < (double)num_nodes_Y))
        return kInf;  // the reference indexes global_layer out of range here
    uint i = (uint)fx, j = (uint)fy;
    double a = x - (double)(i);
    double b = y - (double)(j);
    bool interior = (i + 1 < num_nodes_X) && (j + 1 < num_nodes_Y);
    double w[4] = {kInf, kInf, kInf, kInf};
    if (interior)
    {
        uint32_t idx[4] = {j * num_nodes_X + i, j * num_nodes_X + i + 1, (j + 1) * num_nodes_X + i,
                           (j + 1) * num_nodes_X + i + 1};
        if (!deviceOk(dymu_read_cells(dev, DYMU_PLANE_TOTAL_COST, 0, idx, 4, w), "getTotalCost"))
            return kInf;
    }
    bool all_closed = interior;
    for (int k = 0; k < 4 && all_closed; ++k) all_closed = (w[k] < kInf) && (w[k] <= closed_threshold);
    if (!all_closed)
    {
        long g = nearestIndex(x, y);
        if (g < 0) return kInf;
        uint32_t gi = (uint32_t)g;
        double v = kInf;
        deviceOk(dymu_read_cells(dev, DYMU_PLANE_TOTAL_COST, 0, &gi, 1, &v), "getTotalCost");
        return v;
    }
    double w00 = w[0], w10 = w[1], w01 = w[2], w11 = w[3];
    return w00 + (w10 - w00) * a + (w01 - w00) * b + (w11 + w00 - w10 - w01) * a * b;
}

double DyMuPathPlanner::getTotalCost(base::Waypoint wInt)
{
    return totalCostNoOffset(wInt.position[0] - global_offset[0], wInt.position[1] - global_offset[1]);
}

bool DyMuPathPlanner::getNodeFieldPlane(int field, double* out)
{
    if (!dev || !out) return false;
    size_t n = (size_t)num_nodes_X * num_nodes_Y;
    switch (field)
    {
        case DYMU_NODE_ELEVATION:
            return deviceOk(dymu_download_plane(dev, DYMU_PLANE_ELEVATION, out, num_nodes_X, 0), "tap");
        case DYMU_NODE_SLOPE:
            return deviceOk(dymu_download_plane(dev, DYMU_PLANE_SLOPE, out, num_nodes_X, 0), "tap");
        case DYMU_NODE_RAW_COST:
            return deviceOk(dymu_download_plane(dev, DYMU_PLANE_RAW_COST, out, num_nodes_X, 0), "tap");
        case DYMU_NODE_COST:
            return deviceOk(dymu_download_plane(dev, DYMU_PLANE_COST, out, num_nodes_X, 0), "tap");
        case DYMU_NODE_TOTAL_COST_RAW:
            return deviceOk(dymu_download_total_cost(dev, 0, out, num_nodes_X, 0), "tap");
        case DYMU_NODE_IS_OBSTACLE:
        {
            std::vector<unsigned char> b(n);
            if (!deviceOk(dymu_download_plane_u8(dev, DYMU_PLANE_U8_OBSTACLE, b.data(), num_nodes_X), "tap"))
                return false;
            for (size_t k = 0; k < n; ++k) out[k] = b[k] ? 1.0 : 0.0;
            return true;
        }
        case DYMU_NODE_STATE:
        {
            if (!deviceOk(dymu_download_total_cost(dev, 0, out, num_nodes_X, 0), "tap")) return false;
            for (size_t k = 0; k < n; ++k) out[k] = (out[k] < kInf && out[k] <= closed_threshold) ? 1.0 : 0.0;
            return true;
        }
        case DYMU_NODE_HAS_LOCAL_MAP:
            for (size_t k = 0; k < n; ++k) out[k] = has_local[k] ? 1.0 : 0.0;
            return true;
        default:
            return false;
    }
}

/***********************COST RATIO AFTER TRAVERSE (CoRa)************************/
// reference: G.cpp:895-1038.  The statistics are a few scalars per terrain class and stay on
// the host (DyMuCoRa.hpp); the table they produce feeds the device cost-map kernels again
// through recomputeCostMap().
bool DyMuPathPlanner::initCoRaMethod(int num_terrains_, int num_criteria_, std::vector<double> weights_)
{
    num_terrains = num_terrains_;
    num_criteria = num_criteria_;
    if (cost_lutable.empty() || num_terrains_ < 0 || num_criteria_ < 0) return false;
    base_speed = *std::min_element(cost_lutable.begin(), cost_lutable.end());  // G.cpp:902-904
    if ((int)weights_.size() != num_criteria) return false;
    weights = weights_;
    terrain_vector.resize(num_terrains);
    for (segmentedTerrain& t : terrain_vector)
    {
        t.criteria_info.resize(num_criteria);
        t.traverse_info.resize(num_criteria);
        t.rejected_info.resize(num_criteria);
        t.data_samples.resize(num_criteria);
    }
    return true;
}

int DyMuPathPlanner::getTerrain(base::samples::RigidBodyState current_pos)
{
    base::Pose2D pose;
    pose.position[0] = current_pos.position[0] - global_offset[0];
    pose.position[1] = current_pos.position[1] - global_offset[1];
    globalNode* n = getNearestGlobalNode(pose);
    return n ? (int)n->terrain - 1 : -1;
}
// reference: G.cpp:926-938.  `data` holds one value per criterion, <= 0 meaning "no reading".
bool DyMuPathPlanner::fillTerrainInfo(int terrain_id, std::vector<double> data)
{
    if (terrain_id < 0 || terrain_id >= (int)terrain_vector.size()) return false;  // reference: unchecked
    segmentedTerrain& t = terrain_vector[terrain_id];
    t.dataAnalysis();
    if ((int)data.size() != num_criteria) return false;
    for (int c = 0; c < num_criteria; ++c)
        if (data[c] > 0) t.data_samples[c].push_back(data[c]);
    return true;
}

// reference: G.cpp:956-993.  Chains the pairwise hardness ratios into one relative cost per
// traversed terrain and rewrites locomotion-mode-0 rows of the table for those terrains.
std::vector<double> DyMuPathPlanner::updateCost()
{
    const int range = (int)slope_range.size();
    const int numLocs = (int)locomotion_modes.size();
    for (int t = 0; t < num_terrains && t < (int)terrain_vector.size(); ++t) terrain_vector[t].dataAnalysis();

    std::vector<double> relative(1, 1.0);
    for (double r : computeCostRatio()) relative.push_back(relative.back() / r);
    if (relative.size() < 2) return cost_lutable;
    const double cheapest = *std::min_element(relative.begin(), relative.end());

    size_t rank = 0;  // position of the terrain among the traversed ones
    for (int t = 0; t < num_terrains && t < (int)terrain_vector.size(); ++t)
    {
        if (!terrain_vector[t].traversed) continue;
        // The reference indexes past `relative` when a pair was skipped for lack of common
        // criteria (G.cpp:985) and past the table for terrain ids it does not hold; both stop here.
        if (rank >= relative.size()) break;
        double slope_term = 0;
        for (int s = 0; s < range; ++s)
        {
            slope_term += terrain_vector[t].slope_ratio * slope_range[s];  // cumulative, G.cpp:983
            const size_t idx = (size_t)(t + 1) * range * numLocs + s;
            if (idx < cost_lutable.size()) cost_lutable[idx] = base_speed * relative[rank] / cheapest + slope_term;
        }
        ++rank;
    }
    return cost_lutable;
}

// reference: G.cpp:999-1038.  One ratio per traversed terrain that has a traversed successor.
std::vector<double> DyMuPathPlanner::computeCostRatio()
{
    std::vector<double> cost_ratios;
    const double acc_weight = std::accumulate(weights.begin(), weights.end(), 0.0);
    const int nt = std::min(num_terrains, (int)terrain_vector.size());
    for (int a = 0; a + 1 < nt; ++a)
    {
        if (!terrain_vector[a].traversed) continue;
        int b = a + 1;
        while (b < nt && !terrain_vector[b].traversed) ++b;
        if (b >= nt) continue;
        double hardness_a = 0, hardness_b = 0;
        for (int c = 0; c < num_criteria; ++c)
        {
            const costCriteria &ca = terrain_vector[a].criteria_info[c], &cb = terrain_vector[b].criteria_info[c];
            if (ca.empty || cb.empty) continue;
            hardness_a += weights[c] * ca.mean / acc_weight;
            hardness_b += weights[c] * cb.mean / acc_weight;
        }
        if (hardness_a != 0 && hardness_b != 0) cost_ratios.push_back(hardness_a / hardness_b);
    }
    return cost_ratios;
}

// Extension: apply cost_lutable to the maps resident in HBM (see DyMu.hpp).
bool DyMuPathPlanner::recomputeCostMap(bool resolve)
{
    if (!dev || cost_lutable.empty() || slope_range.empty() || locomotion_modes.empty()) return false;
    if (!deviceOk(dymu_compute_cost_map(dev, cost_lutable.data(), (int)cost_lutable.size(), slope_range.data(),
                                        (int)slope_range.size(), (int)locomotion_modes.size(), NULL, 0, NULL, 0),
                  "recomputeCostMap"))
        return false;
    if (resolve && goal_set) return computeEntireTotalCostMap();
    return true;
}
