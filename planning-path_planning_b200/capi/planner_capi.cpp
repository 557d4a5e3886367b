// planner_capi.cpp -- flat C wrapper over PathPlanning_lib::DyMuPathPlanner.
//
// Contains no planner logic: every function converts arguments to the C++
// types of the class interface (reference: src/DyMu.hpp:471-608), forwards
// the call and converts the result back.  Compiled twice (see
// include/dymu_planner_c.h): with -DDYMU_CAPI_REFERENCE against the
// unmodified reference sources, and with -DDYMU_CAPI_B200 against this
// repository's drop-in DyMu.hpp.  Identical call sequences on both sides are
// what the parity tests rely on.
#include "DyMu.hpp"

#include <chrono>
#include <cstring>
#include <iostream>
#include <mutex>
#include <sstream>
#include <string>
#include <vector>

#include "dymu_planner_c.h"

using PathPlanning_lib::DyMuPathPlanner;

struct dymu_planner
{
    DyMuPathPlanner* impl;
    unsigned nx, ny;
    double last_seconds;
    // arguments of the last computeCostMap, for dymu_planner_recompute_cost_map
    std::vector<double> slopes;
    std::vector<std::string> locs;
#ifdef DYMU_CAPI_REFERENCE
    std::vector<std::vector<double>> elevation, terrain;
#endif
};

namespace
{
// The reference prints progress to std::cout inside the local layer
// (L.cpp:280,584-585,602-608,641-643,680-682).  Silence it unless asked.
// Process-wide and reference-counted: planners may be driven from several threads at once
// (bench.py --impl reference), and swapping std::cout's buffer per call would let one thread
// restore another thread's already destroyed sink.
struct NullBuf : std::streambuf
{
    int overflow(int c) override { return c; }
};
std::mutex g_quiet_mutex;
int g_quiet_depth = 0;
std::streambuf* g_quiet_saved = nullptr;
NullBuf* null_buf()
{
    static NullBuf* b = new NullBuf;  // never destroyed: std::cout may outlive every static here
    return b;
}
struct CoutSilencer
{
    bool active;
    CoutSilencer() : active(!std::getenv("DYMU_CAPI_VERBOSE"))
    {
        if (!active) return;
        std::lock_guard<std::mutex> guard(g_quiet_mutex);
        if (g_quiet_depth++ == 0) g_quiet_saved = std::cout.rdbuf(null_buf());
    }
    ~CoutSilencer()
    {
        if (!active) return;
        std::lock_guard<std::mutex> guard(g_quiet_mutex);
        if (--g_quiet_depth == 0) std::cout.rdbuf(g_quiet_saved);
    }
};

struct Stopwatch
{
    std::chrono::steady_clock::time_point t0;
    double* dst;
    explicit Stopwatch(double* d) : t0(std::chrono::steady_clock::now()), dst(d) {}
    ~Stopwatch()
    {
        *dst = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    }
};

std::vector<std::vector<double>> to_nested(const double* src, unsigned ny, unsigned nx)
{
    std::vector<std::vector<double>> m(ny);
    for (unsigned j = 0; j < ny; ++j) m[j].assign(src + (size_t)j * nx, src + (size_t)(j + 1) * nx);
    return m;
}

void from_nested(const std::vector<std::vector<double>>& m, double* dst)
{
    size_t k = 0;
    for (size_t j = 0; j < m.size(); ++j)
        for (size_t i = 0; i < m[j].size(); ++i) dst[k++] = m[j][i];
}

base::Waypoint make_wp(double x, double y, double heading = 0.0)
{
    base::Waypoint w;
    w.position[0] = x;
    w.position[1] = y;
    w.position[2] = 0.0;
    w.heading = heading;
    return w;
}

int pack_path(const std::vector<base::Waypoint>& path, double* xyzh, int cap)
{
    int n = (int)path.size();
    for (int k = 0; k < n && k < cap; ++k)
    {
        xyzh[4 * k + 0] = path[k].position[0];
        xyzh[4 * k + 1] = path[k].position[1];
        xyzh[4 * k + 2] = path[k].position[2];
        xyzh[4 * k + 3] = path[k].heading;
    }
    return n;
}
}  // namespace

extern "C" {

const char* dymu_planner_impl(void)
{
#if defined(DYMU_CAPI_REFERENCE)
    return "reference";
#else
    return "b200";
#endif
}

dymu_planner* dymu_planner_create(double risk_distance, double reconnect_distance,
                                  double risk_ratio, int approach)
{
    dymu_planner* p = new dymu_planner;
    p->impl = new DyMuPathPlanner(risk_distance, reconnect_distance, risk_ratio,
                                  approach == DYMU_SWEEPING ? PathPlanning_lib::SWEEPING
                                                            : PathPlanning_lib::CONSERVATIVE);
    p->nx = p->ny = 0;
    p->last_seconds = 0.0;
    return p;
}

void dymu_planner_destroy(dymu_planner* p)
{
    if (!p) return;
    delete p->impl;
    delete p;
}

int dymu_planner_init_global_layer(dymu_planner* p, double global_res, double local_res,
                                   unsigned num_nodes_x, unsigned num_nodes_y, double offset_x,
                                   double offset_y)
{
    if (!p) return -1;
    std::vector<double> offset(2);
    offset[0] = offset_x;
    offset[1] = offset_y;
    p->nx = num_nodes_x;
    p->ny = num_nodes_y;
    Stopwatch sw(&p->last_seconds);
    return p->impl->initGlobalLayer(global_res, local_res, num_nodes_x, num_nodes_y, offset) ? 1 : 0;
}

int dymu_planner_set_cost_map(dymu_planner* p, const double* cost, unsigned ny, unsigned nx)
{
    if (!p) return -1;
    std::vector<std::vector<double>> m = to_nested(cost, ny, nx);
    Stopwatch sw(&p->last_seconds);
    return p->impl->setCostMap(m) ? 1 : 0;
}

int dymu_planner_compute_cost_map(dymu_planner* p, const double* cost_data, int n_cost_data,
                                  const double* slope_values, int n_slopes,
                                  const char* locomotion_modes, const double* elevation,
                                  const double* terrain, unsigned ny, unsigned nx)
{
    if (!p) return -1;
    std::vector<double> lut(cost_data, cost_data + n_cost_data);
    std::vector<double> slopes(slope_values, slope_values + n_slopes);
    std::vector<std::string> locs;
    {
        std::stringstream ss(locomotion_modes ? locomotion_modes : "");
        std::string item;
        while (std::getline(ss, item, ',')) locs.push_back(item);
    }
    std::vector<std::vector<double>> e = to_nested(elevation, ny, nx);
    std::vector<std::vector<double>> t = to_nested(terrain, ny, nx);
    p->slopes = slopes;
    p->locs = locs;
#ifdef DYMU_CAPI_REFERENCE
    p->elevation = e;
    p->terrain = t;
#endif
    Stopwatch sw(&p->last_seconds);
    return p->impl->computeCostMap(lut, slopes, locs, e, t) ? 1 : 0;
}

int dymu_planner_recompute_cost_map(dymu_planner* p)
{
    if (!p) return -1;
    Stopwatch sw(&p->last_seconds);
#ifdef DYMU_CAPI_REFERENCE
    if (p->elevation.empty()) return 0;
    return p->impl->computeCostMap(p->impl->cost_lutable, p->slopes, p->locs, p->elevation, p->terrain) ? 1 : 0;
#else
    return p->impl->recomputeCostMap(false) ? 1 : 0;
#endif
}

int dymu_planner_cora_init(dymu_planner* p, int num_terrains, int num_criteria, const double* weights,
                           int n_weights)
{
    if (!p || n_weights < 0) return -1;
    return p->impl->initCoRaMethod(num_terrains, num_criteria,
                                   std::vector<double>(weights, weights + n_weights)) ? 1 : 0;
}

int dymu_planner_get_terrain(dymu_planner* p, double x, double y)
{
    if (!p) return -1;
    base::samples::RigidBodyState rbs;
    rbs.position[0] = x;
    rbs.position[1] = y;
    return p->impl->getTerrain(rbs);
}

int dymu_planner_fill_terrain_info(dymu_planner* p, int terrain_id, const double* data, int n)
{
    if (!p || n < 0) return -1;
    CoutSilencer quiet;
    return p->impl->fillTerrainInfo(terrain_id, std::vector<double>(data, data + n)) ? 1 : 0;
}

int dymu_planner_update_cost(dymu_planner* p, double* lut, int cap)
{
    if (!p) return -1;
    CoutSilencer quiet;
    std::vector<double> v = p->impl->updateCost();
    for (int k = 0; k < (int)v.size() && k < cap; ++k) lut[k] = v[k];
    return (int)v.size();
}

int dymu_planner_compute_cost_ratio(dymu_planner* p, double* ratios, int cap)
{
    if (!p) return -1;
    std::vector<double> v = p->impl->computeCostRatio();
    for (int k = 0; k < (int)v.size() && k < cap; ++k) ratios[k] = v[k];
    return (int)v.size();
}

int dymu_planner_set_goal(dymu_planner* p, double x, double y, double heading)
{
    if (!p) return -1;
    return p->impl->setGoal(make_wp(x, y, heading)) ? 1 : 0;
}

int dymu_planner_compute_total_cost_map(dymu_planner* p, double x, double y)
{
    if (!p) return -1;
    CoutSilencer quiet;
    Stopwatch sw(&p->last_seconds);
    return p->impl->computeTotalCostMap(make_wp(x, y)) ? 1 : 0;
}

int dymu_planner_compute_entire_total_cost_map(dymu_planner* p)
{
    if (!p) return -1;
    CoutSilencer quiet;
    Stopwatch sw(&p->last_seconds);
    return p->impl->computeEntireTotalCostMap() ? 1 : 0;
}

int dymu_planner_get_path(dymu_planner* p, double x, double y, double* xyzh, int cap)
{
    if (!p) return -1;
    CoutSilencer quiet;
    std::vector<base::Waypoint> path;
    {
        Stopwatch sw(&p->last_seconds);
        path = p->impl->getPath(make_wp(x, y));
    }
    return pack_path(path, xyzh, cap);
}

int dymu_planner_compute_global_path(dymu_planner* p, double x, double y)
{
    if (!p) return -1;
    CoutSilencer quiet;
    Stopwatch sw(&p->last_seconds);
    return p->impl->computeGlobalPath(make_wp(x, y)) ? 1 : 0;
}

int dymu_planner_get_current_path(dymu_planner* p, double* xyzh, int cap)
{
    if (!p) return -1;
    return pack_path(p->impl->current_path, xyzh, cap);
}

int dymu_planner_get_matrix(dymu_planner* p, int kind, double* out)
{
    if (!p) return -1;
    std::vector<std::vector<double>> m;
    {
        Stopwatch sw(&p->last_seconds);
        switch (kind)
        {
            case DYMU_MAT_TOTAL_COST: m = p->impl->getTotalCostMatrix(); break;
            case DYMU_MAT_GLOBAL_COST: m = p->impl->getGlobalCostMatrix(); break;
            case DYMU_MAT_HAZARD_DENSITY: m = p->impl->getHazardDensityMatrix(); break;
            case DYMU_MAT_TRAFFICABILITY: m = p->impl->getTrafficabilityMatrix(); break;
            default: return -2;
        }
    }
    from_nested(m, out);
    return 1;
}

double dymu_planner_get_total_cost(dymu_planner* p, double x, double y)
{
    return p->impl->getTotalCost(make_wp(x, y));
}

int dymu_planner_get_locomotion_mode(dymu_planner* p, double x, double y, char* buf, int cap)
{
    if (!p) return -1;
    std::string s = p->impl->getLocomotionMode(make_wp(x, y));
    if ((int)s.size() + 1 > cap) return -2;
    std::memcpy(buf, s.c_str(), s.size() + 1);
    return (int)s.size();
}

int dymu_planner_compute_local_planning(dymu_planner* p, double x, double y,
                                        const uint8_t* image, int w, int h, double res,
                                        double* traj_xyzh, int cap, int* n_traj,
                                        double* local_time_s)
{
    if (!p) return -1;
    CoutSilencer quiet;
    base::samples::frame::Frame frame((uint16_t)w, (uint16_t)h, 1);
    std::memcpy(frame.image.data(), image, (size_t)w * h);
    std::vector<base::Waypoint> traj;
    base::Time t;
    bool ok;
    {
        Stopwatch sw(&p->last_seconds);
        ok = p->impl->computeLocalPlanning(make_wp(x, y), frame, res, traj, t);
    }
    if (n_traj) *n_traj = pack_path(traj, traj_xyzh, cap);
    if (local_time_s) *local_time_s = t.toSeconds();
    return ok ? 1 : 0;
}

int dymu_planner_get_local_matrix(dymu_planner* p, int kind, double x, double y, double* out,
                                  int cap)
{
    if (!p) return -1;
    std::vector<std::vector<double>> m = (kind == DYMU_LOCAL_RISK)
                                             ? p->impl->getRiskMatrix(make_wp(x, y))
                                             : p->impl->getDeviationMatrix(make_wp(x, y));
    int side = (int)m.size();
    if (side * side <= cap) from_nested(m, out);
    return side;
}

int dymu_planner_get_reconnecting_index(dymu_planner* p)
{
    return p->impl->getReconnectingIndex();
}

double dymu_planner_get_remaining_total_cost(dymu_planner* p)
{
    return p->impl->remaining_total_cost;
}

int dymu_planner_get_node_field(dymu_planner* p, int field, double* out)
{
    if (!p) return -1;
#if defined(DYMU_CAPI_B200)
    // The drop-in keeps node fields as device planes; one bulk read-back
    // instead of NX*NY single-node views.
    return p->impl->getNodeFieldPlane(field, out) ? 1 : 0;
#else
    for (unsigned j = 0; j < p->ny; ++j)
        for (unsigned i = 0; i < p->nx; ++i)
        {
            PathPlanning_lib::globalNode* n = p->impl->getGlobalNode(i, j);
            double v = 0.0;
            switch (field)
            {
                case DYMU_NODE_ELEVATION: v = n->elevation; break;
                case DYMU_NODE_SLOPE: v = n->slope; break;
                case DYMU_NODE_RAW_COST: v = n->raw_cost; break;
                case DYMU_NODE_COST: v = n->cost; break;
                case DYMU_NODE_IS_OBSTACLE: v = n->isObstacle ? 1.0 : 0.0; break;
                case DYMU_NODE_STATE: v = (n->state == PathPlanning_lib::CLOSED) ? 1.0 : 0.0; break;
                case DYMU_NODE_HAS_LOCAL_MAP: v = n->hasLocalMap ? 1.0 : 0.0; break;
                case DYMU_NODE_TERRAIN: v = (double)n->terrain; break;
                case DYMU_NODE_TOTAL_COST_RAW: v = n->total_cost; break;
                default: return -2;
            }
            out[(size_t)j * p->nx + i] = v;
        }
    return 1;
#endif
}

int dymu_planner_gradient_node(dymu_planner* p, unsigned i, unsigned j, double* dnx, double* dny)
{
    if (!p || !dnx || !dny) return -1;
    PathPlanning_lib::globalNode* g = p->impl->getGlobalNode(i, j);
    if (!g) return 0;
    p->impl->gradientNode(g, *dnx, *dny);
    return 1;
}

int dymu_planner_next_global_waypoint(dymu_planner* p, double x, double y, double tau, double out[4])
{
    if (!p || !out) return -1;
    base::Waypoint w;
    w.position[0] = x;
    w.position[1] = y;
    base::Waypoint nx = p->impl->computeNextGlobalWaypoint(w, tau);
    out[0] = nx.position[0];
    out[1] = nx.position[1];
    out[2] = nx.heading;
    out[3] = w.position[2];
    return 1;
}

int dymu_planner_propagate_global_node(dymu_planner* p, unsigned i, unsigned j, double* total_cost)
{
    if (!p || !total_cost) return -1;
    PathPlanning_lib::globalNode* g = p->impl->getGlobalNode(i, j);
    if (!g) return 0;
    p->impl->propagateGlobalNode(g);
    *total_cost = g->total_cost;
    return 1;
}

int dymu_planner_set_slope_anisotropy(dymu_planner* p, const double* angles, const double* factors, int n)
{
    if (!p || n < 0 || (n > 0 && (!angles || !factors))) return -1;
#if defined(DYMU_CAPI_B200)
    std::vector<double> a(angles, angles + n), f(factors, factors + n);
    Stopwatch sw(&p->last_seconds);
    return p->impl->setSlopeAnisotropy(a, f) ? 1 : 0;
#else
    return -1;  // the reference's update is isotropic
#endif
}

int dymu_planner_set_obstacle_clearance(dymu_planner* p, double radius, double margin, double penalty)
{
    if (!p) return -1;
#if defined(DYMU_CAPI_B200)
    Stopwatch sw(&p->last_seconds);
    return p->impl->setObstacleClearance(radius, margin, penalty) ? 1 : 0;
#else
    (void)radius;
    (void)margin;
    (void)penalty;
    return -1;  // the reference plans for a point
#endif
}

int dymu_planner_set_cost_map_flat(dymu_planner* p, const double* cost, unsigned ld)
{
    if (!p || !cost || ld < p->nx) return -1;
#if defined(DYMU_CAPI_B200)
    Stopwatch sw(&p->last_seconds);
    return p->impl->setCostMap(cost, (size_t)ld) ? 1 : 0;
#else
    std::vector<std::vector<double>> m(p->ny);
    for (unsigned j = 0; j < p->ny; ++j) m[j].assign(cost + (size_t)j * ld, cost + (size_t)j * ld + p->nx);
    Stopwatch sw(&p->last_seconds);
    return p->impl->setCostMap(m) ? 1 : 0;
#endif
}

int dymu_planner_set_total_cost_target(dymu_planner* p, double* out, unsigned ld)
{
    if (!p || (out && ld < p->nx)) return -1;
#if defined(DYMU_CAPI_B200)
    p->impl->setTotalCostMatrixTarget(out, (size_t)ld);
#endif
    return 1;  // the reference has nothing to prepare
}

int dymu_planner_get_total_cost_matrix_flat(dymu_planner* p, double* out, unsigned ld)
{
    if (!p || !out || ld < p->nx) return -1;
#if defined(DYMU_CAPI_B200)
    Stopwatch sw(&p->last_seconds);
    return p->impl->getTotalCostMatrix(out, (size_t)ld) ? 1 : 0;
#else
    std::vector<std::vector<double>> m;
    {
        Stopwatch sw(&p->last_seconds);
        m = p->impl->getTotalCostMatrix();
    }
    for (unsigned j = 0; j < p->ny; ++j) std::memcpy(out + (size_t)j * ld, m[j].data(), sizeof(double) * p->nx);
    return 1;
#endif
}

double dymu_planner_last_call_seconds(dymu_planner* p) { return p ? p->last_seconds : 0.0; }

}  // extern "C"
