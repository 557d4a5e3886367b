#ifndef _PATHPLANNING_LIBRARIES_HPP_
#define _PATHPLANNING_LIBRARIES_HPP_

// DyMu.hpp -- B200 drop-in for the class interface of ESA-PRL/planning-path_planning.
//
// Same namespace, class name, public method signatures, public data members and return
// conventions as the reference's src/DyMu.hpp:397-609, so that code written against the
// reference library compiles and links against this one.  What is different is where the
// data lives and who does the work:
//
//   * the global layer is not a vector<vector<globalNode*>> of heap nodes but a set of
//     structure-of-arrays planes in B200 HBM, owned by an opaque dymu_ctx
//     (include/dymu_cuda.h); every wave propagation, stencil and path descent runs in
//     hand-written sm_100a kernels behind that C ABI;
//   * the local layer is a dense device window instead of lazily linked localNodes;
//   * this class keeps only the sequential control logic of the reference on the host
//     (goal/start validation, repairPath / evaluatePath splicing, index bookkeeping).
//
// globalNode / localNode are kept as plain value "views": getGlobalNode()/getLocalNode()
// fill one from the device planes on request.  Their neighbour lists are empty (no
// pointer graph exists any more).  The CoRa cost-ratio learning methods
// (src/DyMu.hpp:593-608) keep their scalar statistics on the host (DyMuCoRa.hpp); the table
// they produce is applied on the device by recomputeCostMap().
//
// There is no CPU fallback: without a CUDA device initGlobalLayer returns false.

#include <base/Waypoint.hpp>
#include <base/samples/Frame.hpp>
#include <base/samples/RigidBodyState.hpp>
#include <map>
#include <numeric>
#include <string>
#include <vector>

#include <base-logging/Logging.hpp>

#include "DyMuCoRa.hpp"

struct dymu_ctx;

namespace PathPlanning_lib
{
enum node_state
{
    OPEN,
    CLOSED
};

enum repairingAproach
{
    CONSERVATIVE,  // Hazard Avoidance - FM*
    SWEEPING       // multiBiFM*
};

// Value view of one local node (reference: src/DyMu.hpp:42-67).
struct localNode
{
    base::Pose2D pose;         // In Local Units respect to Global Node
    base::Pose2D world_pose;   // In physical Units respect to World Frame
    base::Pose2D parent_pose;  // Position of Global Node Parent In Global Units
    base::Pose2D global_pose;  // Position of this local node in Global Units
    double deviation;
    double total_cost;
    double cost;
    double risk;
    node_state state;
    std::vector<localNode*> nb4List;  // always empty in this build
    bool isObstacle;
    long window_cell;  // index inside the device window (-1 = outside)
    localNode() : deviation(0), total_cost(0), cost(0), risk(0), state(OPEN), isObstacle(false), window_cell(-1) {}
};

// Value view of one global node (reference: src/DyMu.hpp:69-108).
struct globalNode
{
    base::Pose2D pose;
    base::Pose2D world_pose;
    double elevation;
    double slope;
    node_state state;
    bool isObstacle;
    bool hasLocalMap;
    double raw_cost;
    double cost;
    double hazard_density;
    double trafficability;
    double total_cost;
    unsigned int terrain;
    std::vector<std::vector<localNode*>> localMap;  // always empty in this build
    std::vector<globalNode*> nb4List;                // always empty in this build
    std::vector<globalNode*> nb8List;                // always empty in this build
    std::string nodeLocMode;
    globalNode()
        : elevation(0), slope(0), state(OPEN), isObstacle(false), hasLocalMap(false), raw_cost(0),
          cost(0), hazard_density(0), trafficability(1), total_cost(0), terrain(0),
          nodeLocMode("DONT_CARE")
    {
    }
};

//__DYMU_PATH_PLANNER_CLASS__
class DyMuPathPlanner
{
  private:
    // device side
    dymu_ctx* dev;
    // Dimensions
    uint num_nodes_X;
    uint num_nodes_Y;
    double global_res;
    std::vector<double> global_offset;
    double local_res;
    uint res_ratio;

    // Local Repairing Parameters
    double risk_distance;
    double reconnect_distance;
    double risk_ratio;
    std::vector<double> slope_range;
    std::vector<std::string> locomotion_modes;
    repairingAproach repairing_approach;

    // CoRa state (reference: src/DyMu.hpp:429-439)
    std::vector<segmentedTerrain> terrain_vector;
    std::vector<double> weights;
    int num_terrains;
    int num_criteria;
    double base_speed;

    // host-side layer bookkeeping (bit-exact emulation of hasLocalMap, DyMu.hpp:77)
    std::vector<unsigned char> has_local;
    // goal
    bool goal_set;
    uint goal_i, goal_j;
    // CLOSED-set emulation: a node is CLOSED iff total_cost <= closed_threshold
    double closed_threshold;
    // total-cost matrix delivery started right after a solve (setTotalCostMatrixTarget)
    double* readback_target;
    size_t readback_ld;
    bool readback_inflight;
    bool streamed_cost;  // the last cost-map call was a streamed setCostMap(const double*, ld)
    double clearance_radius;  // lethal radius of the obstacle clearance in effect (0: none)
    // obstacles ingested but not yet expanded (local_expandable_obstacles, DyMu.hpp:452)
    bool pending_risk;
    uint local_window_nodes;
    bool local_ready;    // the window is placed (anchored) and holds the local layer
    bool local_created;  // the window is allocated
    long local_agent_cell;
    // node views handed out by getGlobalNode / getLocalNode
    std::map<unsigned long long, globalNode> global_views;
    std::map<long, localNode> local_views;
    globalNode goal_view;
    localNode agent_view;
    std::string last_error;

    // helpers (not part of the reference interface)
    bool deviceOk(int rc, const char* what);
    long nearestIndex(double x, double y) const;  // getNearestGlobalNode as j*NX+i or -1
    void subdivideIndex(long g);
    bool ensureLocalWindow(double x, double y, double half_x, double half_y, bool may_grow);
    bool growLocalWindow(long lo_x, long hi_x, long lo_y, long hi_y);
    bool readNode(uint i, uint j, globalNode& out);
    bool goalInLethalRing();
    void markEntered();
    long localPropagationCell(base::Waypoint wInit, base::Waypoint wOvertake);
    std::vector<base::Waypoint> localPathFromCell(long cell, base::Waypoint wInit);
    void localCellPose(long cell, double& gx, double& gy) const;
    double totalCostNoOffset(double x, double y);
    long viewCell(localNode* n);
    void startReadback();
    void finishReadback();

  public:
    // -- PARAMETERS -- (kept for source compatibility; the narrow bands are transient
    // state of the sequential algorithm and stay empty here)
    std::vector<globalNode*> global_narrowband;
    std::vector<globalNode*> global_propagated_nodes;
    std::vector<localNode*> local_narrowband;
    std::vector<localNode*> local_expandable_obstacles;
    std::vector<localNode*> local_propagated_nodes;
    // The last computed path
    std::vector<base::Waypoint> current_path;
    // LookUp Table containing cost values per terrain and slope value
    std::vector<double> cost_lutable;
    // Global Node containing the goal
    globalNode* global_goal;
    // Local Node containing the position of the agent
    localNode* local_agent;
    // Total Cost needed by the agent to reach the goal
    double remaining_total_cost;
    // Index to current path in which the local path meets global
    int reconnecting_index;

    // -- FUNCTIONS --
    DyMuPathPlanner(double risk_distance,
                    double reconnect_distance,
                    double risk_ratio,
                    repairingAproach input_approach);
    ~DyMuPathPlanner();

    bool initGlobalLayer(double globalres,
                         double localres,
                         uint num_nodes_X,
                         uint num_nodes_Y,
                         std::vector<double> offset);

    bool setCostMap(std::vector<std::vector<double>> cost_map);

    bool computeCostMap(std::vector<double> cost_data,
                        std::vector<double> slope_values,
                        std::vector<std::string> locomotionModes,
                        std::vector<std::vector<double>> elevation,
                        std::vector<std::vector<double>> terrainMap);

    // Node-level steps (reference: H.hpp:497-575), forwards onto value views: DyMuNodeLevel.cpp
    void calculateSlope(globalNode* nodeTarget);
    void calculateNominalCost(globalNode* nodeTarget, int range, int numLocs);
    void smoothCost(globalNode* nodeTarget);

    // Returns a view of global node (i,j), NULL if out of range
    globalNode* getGlobalNode(uint i, uint j);

    bool setGoal(base::Waypoint wGoal);

    bool computeTotalCostMap(base::Waypoint wPos);
    bool computeEntireTotalCostMap();

    bool isSafeNode(globalNode* global_node);
    bool isFullyClosedNode(globalNode* global_node);

    void resetTotalCostMap();
    void resetGlobalNarrowBand();

    void propagateGlobalNode(globalNode* nodeTarget);
    globalNode* minCostGlobalNode();

    globalNode* getNearestGlobalNode(base::Pose2D pos);
    globalNode* getNearestGlobalNode(base::Waypoint wPos);

    std::vector<base::Waypoint> getPath(base::Waypoint wPos);

    bool computeGlobalPath(base::Waypoint wPos);

    base::Waypoint computeNextGlobalWaypoint(base::Waypoint& wPos, double tau);
    void gradientNode(globalNode* nodeTarget, double& dnx, double& dny);

    double interpolate(double a, double b, double g00, double g01, double g10, double g11);

    std::string getLocomotionMode(base::Waypoint wPos);

    std::vector<std::vector<double>> getTotalCostMatrix();
    std::vector<std::vector<double>> getGlobalCostMatrix();
    std::vector<std::vector<double>> getHazardDensityMatrix();
    std::vector<std::vector<double>> getTrafficabilityMatrix();

    double getTotalCost(base::Waypoint wInt);

    // LOCAL PATH REPAIRING
    void createLocalMap(globalNode* gNode);
    localNode* getLocalNode(base::Pose2D pos);
    localNode* getLocalNode(base::Waypoint wPos);

    void subdivideGlobalNode(globalNode* gNode);

    bool computeLocalPlanning(base::Waypoint wPos,
                              base::samples::frame::Frame traversabilityMap,
                              double res,
                              std::vector<base::Waypoint>& trajectory,
                              base::Time& localTime);

    void expandRisk();
    localNode* maxRiskNode();
    void propagateRisk(localNode* nodeTarget);
    void setHorizonCost(localNode* horizonNode);

    double getTotalCost(localNode* lNode);

    localNode* computeLocalPropagation(base::Waypoint wInit, base::Waypoint wOvertake);
    void propagateLocalNode(localNode* nodeTarget);
    localNode* minCostLocalNode(double Tovertake, double minC);
    localNode* minCostLocalNode(localNode* reachNode);

    std::vector<base::Waypoint> getLocalPath(localNode* lSetNode, base::Waypoint wInit, double tau);

    bool computeLocalWaypointGDM(base::Waypoint& wPos, double tau);
    base::Waypoint computeLocalWaypointDijkstra(localNode* lNode);
    void gradientNode(localNode* nodeTarget, double& dnx, double& dny);

    bool evaluatePath(uint starting_index);
    bool isBlockingObstacle(localNode* obNode, uint& maxIndex, uint& minIndex);

    int repairPath(base::Waypoint wInit, uint index);

    std::vector<std::vector<double>> getRiskMatrix(base::Waypoint rover_pos);
    std::vector<std::vector<double>> getDeviationMatrix(base::Waypoint rover_pos);

    int getReconnectingIndex();

    // COST RATIO UPDATING AFTER TRAVERSE (CoRa), reference: G.cpp:895-1038
    bool initCoRaMethod(int num_terrains_, int num_criteria_, std::vector<double> weights_);
    int getTerrain(base::samples::RigidBodyState current_pos);
    bool fillTerrainInfo(int terrain_id, std::vector<double> data);
    std::vector<double> updateCost();
    std::vector<double> computeCostRatio();

    // ---- extensions of this build (not in the reference) --------------------------------
    // flat, copy-free variants of the map setters (row-major [j][i], ld doubles per row)
    bool setCostMap(const double* cost_map, size_t ld);
    bool computeCostMap(const std::vector<double>& cost_data, const std::vector<double>& slope_values,
                        const std::vector<std::string>& locomotionModes, const double* elevation,
                        size_t ld_e, const double* terrainMap, size_t ld_t);
    bool getTotalCostMatrix(double* out, size_t ld);
    // Deliver the total-cost matrix into `out` (row-major, ld doubles per row, pinned memory for a
    // truly asynchronous copy) right after every successful compute*TotalCostMap, overlapped with
    // the caller's next calls; getTotalCostMatrix(out, ld) then only waits.  NULL = off.
    void setTotalCostMatrixTarget(double* out, size_t ld);
    // Apply the current cost_lutable (e.g. the one updateCost() just produced) to the DEM and
    // terrain classes that are already resident in HBM -- the reference's caller would hand
    // both maps to computeCostMap again.  With resolve=true and a goal set, the total-cost
    // map is recomputed as well.
    bool recomputeCostMap(bool resolve = false);
    // Slope anisotropy for every later compute*TotalCostMap, getPath and computeGlobalPath: the
    // cost of moving from a node to a 4-neighbour is its cost term times f(theta), theta the
    // signed slope angle toward that neighbour in degrees (positive = uphill) and f piecewise
    // linear in (slope_angles_deg, factors), clamped at both ends (DESIGN.md section 10).  Angles
    // strictly ascending, factors finite > 0, at least two pairs; empty vectors switch it off.
    // False before initGlobalLayer and on a malformed table.  The local layer stays isotropic.
    bool setSlopeAnisotropy(const std::vector<double>& slope_angles_deg, const std::vector<double>& factors);
    // Obstacle clearance for every later compute*TotalCostMap, getPath and computeGlobalPath (metres;
    // DESIGN.md section 11): nodes within `radius` of an obstacle node become impassable (the lethal
    // ring; the obstacle map itself is unchanged), the cost of nodes between radius and
    // radius + margin is scaled by 1 + penalty * (radius + margin - d) / margin, d the distance to the
    // nearest obstacle node.  radius = margin = 0 switches it off.  A goal inside the lethal ring is
    // not valid, like a goal on an obstacle.  False before initGlobalLayer and on a malformed setting
    // (negative or non-finite values, radius + margin over 128 global nodes).  The local layer keeps
    // its own risk dilation.
    bool setObstacleClearance(double radius, double margin, double penalty);
    // read-only view of the CoRa accumulators (test tap)
    const std::vector<segmentedTerrain>& terrainInfo() const { return terrain_vector; }
    // bulk tap of one globalNode field (DYMU_NODE_* of include/dymu_planner_c.h)
    bool getNodeFieldPlane(int field, double* out);
    // size of the dense local window in global nodes (default 64)
    void setLocalWindow(uint nodes) { local_window_nodes = nodes; }
    dymu_ctx* deviceContext() { return dev; }
    const std::string& lastError() const { return last_error; }
};

}  // namespace PathPlanning_lib

#endif  // _PATHPLANNING_LIBRARIES_HPP_
