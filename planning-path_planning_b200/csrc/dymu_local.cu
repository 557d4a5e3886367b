// dymu_local.cu -- the local (fine) layer of DyMu on the device
// (reference: src/DyMu_LocalPathRepairing.cpp, "L.cpp").
//
// The reference subdivides global nodes lazily into res_ratio x res_ratio localNodes linked
// by pointers (L.cpp:23-156).  Here the local layer is a dense window of wg x wg global
// nodes around the rover: SoA planes risk / deviation / total_cost / isObstacle / state,
// window cell (X, Y) <-> local node (li, lj) = (X % r, Y % r) of global node
// (gx0 + X / r, gy0 + Y / r).  A missing link (NULL) in the reference can only occur
// across the border of the global map, because every node the waves touch has had its
// parent and the parent's 8 neighbours subdivided first (L.cpp:166,182,505-507,660-662).
//
// Kernels:
//   k_ingest_*       obstacle/risk mask from the traversability frame   (L.cpp:233-259)
//   k_blocking       isBlockingObstacle as a parallel min/max reduction (L.cpp:441-471)
//   risk dilation    MODE 1 of the tiled FIM kernel (dymu_fim.cu)       (L.cpp:493-576)
//   k_local_march    narrow-band march on `deviation` in the reference's exact pop order,
//                    two warps: order-preserving erase and the four neighbour updates on
//                    four lanes of warp 0, the argmin scan of the band on warp 1 one pop
//                    ahead                                              (L.cpp:578-805)
//   k_local_path     single-warp gradient descent with Dijkstra fallback (L.cpp:807-1023)
#include <stdlib.h>

#include "dymu_ctx.cuh"

int dymu_internal_fill(dymu_ctx* ctx, double* p, double v, size_t n);

#include <algorithm>
#include <chrono>
#include <cstdio>

namespace
{
constexpr uint32_t kNoCell = 0xFFFFFFFFu;

// DYMU_TRACE_CALLS=1: wall time of every local-layer entry point on stderr (developer aid)
struct CallTrace
{
    const char* name;
    std::chrono::steady_clock::time_point t0;
    bool on;
    explicit CallTrace(const char* n) : name(n), on(getenv("DYMU_TRACE_CALLS") != nullptr)
    {
        if (on) t0 = std::chrono::steady_clock::now();
    }
    ~CallTrace()
    {
        if (on)
            fprintf(stderr, "[dymu] %-28s %9.3f ms\n", name,
                    std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    }
};

struct LocalView
{
    double *risk, *dev, *ltot;
    uint8_t *obst, *state;
    uint32_t w, pitch, r;       // window edge (cells), row pitch, cells per global node edge
    int64_t gx0, gy0;           // anchor global node
    uint32_t nx, ny;            // global grid
    double gres, lres;
    const double* T;            // global total cost (slot 0)
    const double* elev;
    const uint8_t* gobst;
    uint32_t gpitch;
};

__device__ __forceinline__ bool global_node_of(const LocalView& v, double x, double y, int64_t& gi,
                                               int64_t& gj)
{
    // getNearestGlobalNode, G.cpp:572-584 (negative -> unsigned wrap -> NULL)
    double fx = x / v.gres + 0.5, fy = y / v.gres + 0.5;
    if (!(fx >= 0.0) || !(fy >= 0.0) || !(fx < 4294967296.0) || !(fy < 4294967296.0)) return false;
    uint32_t ui = (uint32_t)fx, uj = (uint32_t)fy;
    if (ui >= v.nx || uj >= v.ny) return false;
    gi = ui;
    gj = uj;
    return true;
}

// getLocalNode, L.cpp:160-189 -> window cell; kNoCell-like (-1) when outside map, -2 when
// inside the map but outside the window
__device__ __forceinline__ int64_t cell_of(const LocalView& v, double x, double y)
{
    int64_t gi, gj;
    if (!global_node_of(v, x, y, gi, gj)) return -1;
    double cornerX = (double)gi - v.gres / 2, cornerY = (double)gj - v.gres / 2;
    double a = x - cornerX, b = y - cornerY;
    uint32_t li = (uint32_t)(a * v.r), lj = (uint32_t)(b * v.r);
    if (li >= v.r) li = v.r - 1;  // reference would index out of bounds
    if (lj >= v.r) lj = v.r - 1;
    int64_t X = (gi - v.gx0) * (int64_t)v.r + li, Y = (gj - v.gy0) * (int64_t)v.r + lj;
    if (X < 0 || Y < 0 || X >= (int64_t)v.w || Y >= (int64_t)v.w) return -2;
    return Y * (int64_t)v.w + X;
}

__device__ __forceinline__ void cell_xy(const LocalView& v, int64_t c, uint32_t& X, uint32_t& Y)
{
    X = (uint32_t)(c % v.w);
    Y = (uint32_t)(c / v.w);
}
__device__ __forceinline__ size_t cell_addr(const LocalView& v, int64_t c)
{
    return (size_t)(c / v.w) * v.pitch + (size_t)(c % v.w);
}
// localNode::global_pose, L.cpp:35-40
__device__ __forceinline__ void global_pose(const LocalView& v, int64_t c, double& gx, double& gy)
{
    uint32_t X, Y;
    cell_xy(v, c, X, Y);
    double px = (double)(v.gx0 + X / v.r), py = (double)(v.gy0 + Y / v.r);
    double lx = (double)(X % v.r), ly = (double)(Y % v.r), rr = (double)v.r;
    gx = px - 0.5 + (0.5 / rr) + lx * (1 / rr);
    gy = py - 0.5 + (0.5 / rr) + ly * (1 / rr);
}
// localNode::world_pose, L.cpp:41-44
__device__ __forceinline__ void world_pose(const LocalView& v, int64_t c, double& wx, double& wy)
{
    double gx, gy;
    global_pose(v, c, gx, gy);
    wx = gx / v.gres;
    wy = gy / v.gres;
}
// parent as the reference finds it: getNearestGlobalNode(parent_pose), i.e. the parent's
// node coordinates divided by global_res once more (quirk 4 of SURVEY.md section 2.2)
__device__ __forceinline__ bool parent_via_nearest(const LocalView& v, int64_t c, int64_t& gi,
                                                   int64_t& gj)
{
    uint32_t X, Y;
    cell_xy(v, c, X, Y);
    return global_node_of(v, (double)(v.gx0 + X / v.r), (double)(v.gy0 + Y / v.r), gi, gj);
}

// neighbour in nb4List order (L.cpp:57-65): 0 (Y-1), 1 (X-1), 2 (X+1), 3 (Y+1).
// returns -1: NULL (outside the global map); -2: inside the map but outside the window
__device__ __forceinline__ int64_t lnb4(const LocalView& v, int64_t c, int d)
{
    if (c < 0) return -1;
    int64_t X = c % v.w, Y = c / v.w;
    if (d == 0) Y -= 1; else if (d == 1) X -= 1; else if (d == 2) X += 1; else Y += 1;
    int64_t LX = v.gx0 * (int64_t)v.r + X, LY = v.gy0 * (int64_t)v.r + Y;
    if (LX < 0 || LY < 0 || LX >= (int64_t)v.nx * v.r || LY >= (int64_t)v.ny * v.r) return -1;
    if (X < 0 || Y < 0 || X >= (int64_t)v.w || Y >= (int64_t)v.w) return -2;
    return Y * (int64_t)v.w + X;
}

// ---------------------------------------------------------------------------------
// obstacle ingestion
// ---------------------------------------------------------------------------------
struct IngestArgs
{
    LocalView v;
    const uint8_t* image;
    uint32_t w, h, row_size, pixel_size;
    double res, rover_x, rover_y;
    uint32_t* first;     // per window cell: lowest qualifying pixel index
    uint32_t* winner;    // per pixel: window cell it newly marks, or kNoCell
    uint32_t* flags;     // [0] window exceeded
};

__device__ __forceinline__ int64_t pixel_cell(const IngestArgs& a, uint32_t p, bool& qualifies)
{
    qualifies = false;
    uint32_t j = p / a.w, i = p % a.w;
    // L.cpp:225-241 (image convention, Y pointing down)
    double offsetX = a.rover_x - a.res * (double)a.w / 2;
    double offsetY = a.rover_y + a.res * (double)a.h / 2;
    double globalSizeX = a.v.gres * (double)a.v.nx - 0.5, globalSizeY = a.v.gres * (double)a.v.ny - 0.5;
    double px = offsetX + i * a.res, py = offsetY - j * a.res;
    if (!((px > -0.5) && (px < globalSizeX) && (py > -0.5) && (py < globalSizeY))) return -1;
    int64_t c = cell_of(a.v, px, py);
    if (c == -2) { a.flags[0] = 1; return -2; }
    if (c < 0) return -1;
    uint8_t value = a.image[(size_t)j * a.row_size + (size_t)i * a.pixel_size];
    int64_t gi, gj;
    bool gob = false;
    if (parent_via_nearest(a.v, c, gi, gj)) gob = a.v.gobst[(size_t)gj * a.v.gpitch + gi] != 0;
    qualifies = (!a.v.obst[cell_addr(a.v, c)]) && ((value != 0) || gob);  // L.cpp:250
    return c;
}

__global__ void k_ingest_claim(IngestArgs a)
{
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.w * a.h) return;
    bool q;
    int64_t c = pixel_cell(a, p, q);
    if (c >= 0 && q) atomicMin(&a.first[c], p);
}

__global__ void k_ingest_mark(IngestArgs a)
{
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.w * a.h) return;
    bool q;
    int64_t c = pixel_cell(a, p, q);
    uint32_t win = kNoCell;
    if (c >= 0 && q && a.first[c] == p) win = (uint32_t)c;
    a.winner[p] = win;
}

// second phase so that k_ingest_mark still sees the pre-ingest obstacle mask
__global__ void k_ingest_commit(IngestArgs a)
{
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.w * a.h) return;
    uint32_t c = a.winner[p];
    if (c != kNoCell)
    {
        size_t q = cell_addr(a.v, c);
        a.v.obst[q] = 1;     // L.cpp:257
        a.v.risk[q] = 1.0;   // L.cpp:259
    }
}

// ---------------------------------------------------------------------------------
// isBlockingObstacle, L.cpp:441-471: per obstacle the first in-range waypoint index feeds
// minIndex, and the index at which the path leaves the range (or path.size()) feeds maxIndex
// ---------------------------------------------------------------------------------
// One warp per obstacle cell, the lanes stride over the waypoints; the sequential scan of the
// reference becomes "first in-range index f" and "first out-of-range index after f".
__global__ void k_blocking(LocalView v, const uint32_t* cells, uint32_t n_cells,
                           const double* path_xy, uint32_t n_path, double risk_distance,
                           uint32_t* out /* [0] min, [1] max, [2] blocked */)
{
    const unsigned full = 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (k >= n_cells) return;  // warp-uniform
    double wx, wy;
    world_pose(v, cells[k], wx, wy);
    bool blocked = false, left_range = false;
    uint32_t mn = 0xFFFFFFFFu, mx = 0;
    for (uint32_t base = 0; base < n_path && !left_range; base += 32)
    {
        const uint32_t i = base + lane;
        bool in_range = false;
        if (i < n_path)
        {
            double dx = wx - path_xy[2 * i], dy = wy - path_xy[2 * i + 1];
            in_range = sqrt(dx * dx + dy * dy) < risk_distance;
        }
        const unsigned valid = (n_path - base >= 32) ? full : ((1u << (n_path - base)) - 1);
        const unsigned m = __ballot_sync(full, in_range);
        unsigned after = valid;  // positions where leaving the range counts
        if (!blocked)
        {
            if (!m) continue;
            const uint32_t f = __ffs(m) - 1;
            blocked = true;
            mn = base + f;
            after &= (f == 31) ? 0u : (full << (f + 1));
        }
        const unsigned leave = ~m & after;
        if (leave)
        {
            mx = base + __ffs(leave) - 1;
            left_range = true;
        }
    }
    if (blocked && !left_range) mx = n_path;  // L.cpp:467-468
    if (blocked && lane == 0)
    {
        atomicMin(&out[0], mn);
        atomicMax(&out[1], mx);
        out[2] = 1;
    }
}

// C plane of the risk dilation: constant local_res / risk_distance (L.cpp:562); obstacle
// cells and padding are never targets (L.cpp:503, 509)
__global__ void k_risk_cplane(const uint8_t* obst, double* crisk, double C, uint32_t pitch,
                              uint32_t rows, uint32_t w)
{
    size_t total = (size_t)pitch * rows;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += stride)
    {
        uint32_t y = (uint32_t)(q / pitch), x = (uint32_t)(q % pitch);
        crisk[q] = (x < w && y < w && !obst[q]) ? C : DYMU_INF;
    }
}

// Which global nodes would the reference have subdivided while dilating risk?  Every node
// holding a popped cell (risk > 0) and every node holding a non-obstacle 4-neighbour of one
// (expandRisk looks at the neighbour's parent before propagating, L.cpp:501-510).
__global__ void k_mark_entered_risk(LocalView v, uint8_t* entered)
{
    size_t total = (size_t)v.w * v.w;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    uint32_t wg = v.w / v.r;
    for (size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x; c < total; c += stride)
    {
        if (!(v.risk[cell_addr(v, (int64_t)c)] > 0)) continue;
        uint32_t X, Y;
        cell_xy(v, (int64_t)c, X, Y);
        entered[(Y / v.r) * wg + X / v.r] = 1;
        for (int d = 0; d < 4; ++d)
        {
            int64_t nb = lnb4(v, (int64_t)c, d);
            if (nb < 0 || v.obst[cell_addr(v, nb)]) continue;
            uint32_t NX_, NY_;
            cell_xy(v, nb, NX_, NY_);
            entered[(NY_ / v.r) * wg + NX_ / v.r] = 1;
        }
    }
}

// ---------------------------------------------------------------------------------
// local propagation in the reference's pop order
// ---------------------------------------------------------------------------------
struct MarchArgs
{
    LocalView v;
    int approach;            // 0 CONSERVATIVE, 1 SWEEPING
    double sx, sy, ox, oy;   // start / overtake waypoint (offset-free)
    double t_overtake, risk_ratio;
    uint32_t* nb;            // per window cell: narrow-band slot of the node (see k_local_march)
    uint32_t* prop;          // local_propagated_nodes
    uint32_t cap;
    uint8_t* entered;        // per window global node: the wave looked into it (L.cpp:660-662)
    int64_t* result;         // [0] end cell [1] status [2] closed [3] prop count [4] nb peak
    const double* ltot_cache; // getTotalCost of every window cell (k_local_total_cost_cache)
    uint32_t prev_prop;      // nodes to reset from the previous call (L.cpp:589-599)
    uint64_t max_pops;
    // per-axis tables the march fills before its first pop (everything in them depends on one
    // window coordinate only): squared world distance to the end node per column / row
    // (CONSERVATIVE key, L.cpp:735-741) and the node getNearestGlobalNode maps a parent to
    double* axis_d2;         // [2 * w]: columns, then rows
    int32_t* axis_node;      // [2 * wg]: columns, then rows; -1: no node
};

// getTotalCost(localNode*), L.cpp:473-491
__device__ __forceinline__ double local_total_cost(const LocalView& v, int64_t c)
{
    double gx, gy;
    global_pose(v, c, gx, gy);
    uint32_t i = (uint32_t)gx, j = (uint32_t)gy;
    double a = gx - (double)i, b = gy - (double)j;
    int64_t gi, gj;
    const double inf = DYMU_INF;
    if (!parent_via_nearest(v, c, gi, gj)) return inf;  // reference dereferences NULL
    double w00 = v.T[(size_t)gj * v.gpitch + gi];
    double w10 = (gi + 1 < (int64_t)v.nx) ? v.T[(size_t)gj * v.gpitch + gi + 1] : inf;
    double w01 = (gj + 1 < (int64_t)v.ny) ? v.T[(size_t)(gj + 1) * v.gpitch + gi] : inf;
    double w11 = (gi + 1 < (int64_t)v.nx && gj + 1 < (int64_t)v.ny)
                     ? v.T[(size_t)(gj + 1) * v.gpitch + gi + 1] : inf;
    return w00 + (w10 - w00) * a + (w01 - w00) * b + (w11 + w00 - w10 - w01) * a * b;
}

// The narrow band lives in shared memory as an append-only array of (cell, key) slots:
//   * push_back  -> append at `tail`
//   * erase(k)   -> the slot becomes a tombstone (key = +inf); relative order of the survivors,
//                   which is what the reference's strict '<' scan breaks ties by, is untouched
//   * a lowered deviation of a node that is already in the band rewrites its cached key through
//     the per-cell slot map `pos`
//   * the array is compacted (stable) when it runs full or mostly holds tombstones.
// Keys of live slots are finite, so +inf is free to mean "erased".
constexpr uint32_t kBandSlots = 12288;
static_assert(kBandSlots < (1u << 14), "k_local_march packs slot numbers into 14 bits");
constexpr size_t kBandSmem = (size_t)kBandSlots * (sizeof(double) + sizeof(uint32_t));

// 0: usable cell; -1: outside the global map (NULL in the reference); -2: outside the window
__device__ __forceinline__ int cell_class(const LocalView& v, int64_t bx, int64_t by, int X, int Y)
{
    int64_t LX = bx + X, LY = by + Y;
    if (LX < 0 || LY < 0 || LX >= (int64_t)v.nx * v.r || LY >= (int64_t)v.ny * v.r) return -1;
    if (X < 0 || Y < 0 || X >= (int)v.w || Y >= (int)v.w) return -2;
    return 0;
}

struct MapBox
{
    int x0, x1, y0, y1, w;
};
__device__ __forceinline__ int clamp_box(int64_t t, uint32_t w)
{
    return (int)max((int64_t)-4, min(t, (int64_t)w + 4));
}
// same classes as cell_class for window coordinates within one step of the window
__device__ __forceinline__ int box_class(const MapBox& b, int X, int Y)
{
    if (X < b.x0 || X >= b.x1 || Y < b.y0 || Y >= b.y1) return -1;
    if ((unsigned)X >= (unsigned)b.w || (unsigned)Y >= (unsigned)b.w) return -2;
    return 0;
}

// world_pose (L.cpp:35-44) from window coordinates, same expression order as global_pose()
__device__ __forceinline__ double world_axis(const LocalView& v, int64_t g0, uint32_t X)
{
    double px = (double)(g0 + X / v.r);
    double lx = (double)(X % v.r), rr = (double)v.r;
    return (px - 0.5 + (0.5 / rr) + lx * (1 / rr)) / v.gres;
}
__device__ __forceinline__ void world_xy(const LocalView& v, uint32_t X, uint32_t Y, double& wx, double& wy)
{
    wx = world_axis(v, v.gx0, X);
    wy = world_axis(v, v.gy0, Y);
}
// one axis of getNearestGlobalNode (G.cpp:572-584) for node coordinate g: the node index or -1
__device__ __forceinline__ int32_t nearest_node_axis(double gres, double g, uint32_t n)
{
    double f = g / gres + 0.5;
    if (!(f >= 0.0) || !(f < 4294967296.0)) return -1;
    uint32_t u = (uint32_t)f;
    return u >= n ? -1 : (int32_t)u;
}

// propagateLocalNode's neighbour pair rule, L.cpp:705-717 (ca/cb: cell_class of the pair)
__device__ __forceinline__ double dev_pair(const double* D, int ca, size_t oa, int cb, size_t ob)
{
    if (ca == 0 && cb == 0) return fmin(D[ob], D[oa]);
    if (ca != 0) return (cb == 0) ? D[ob] : DYMU_INF;
    return D[oa];
}

// getTotalCost(localNode*) for every window cell at once.  The march copies a value into the
// node's total_cost the first time the wave looks at it (L.cpp:666-667), so that the lazily
// filled plane the reference exposes stays the same while the march itself never waits for the
// global total-cost plane.
__global__ void k_local_total_cost_cache(LocalView v, double* cache)
{
    size_t total = (size_t)v.w * v.w;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x; c < total; c += stride)
    {
        uint32_t X = (uint32_t)(c % v.w), Y = (uint32_t)(c / v.w);
        cache[(size_t)Y * v.pitch + X] = local_total_cost(v, (int64_t)c);
    }
}

// Two warps.  Warp 0 is the march: pop, erase, the four neighbour updates, push -- strictly in the
// reference's order.  Warp 1 only looks for minima: as soon as warp 0 has announced which slot pop
// k takes, warp 1 scans the band for the best of the REST (keys as they were before pop k touched
// anything) while warp 0 updates the neighbours.  Keys only ever decrease and new entries only
// appear at the tail, so the minimum for pop k+1 is the lexicographic (key, slot) minimum of that
// "best of the rest" and the at most four entries pop k lowered or created -- which warp 0 holds
// in registers.  The band scan, 40 % of a pop, leaves the critical path.
constexpr unsigned long long kMarchExit = ~0ull;
constexpr int kMarchSpinLimit = 1 << 26;  // a broken hand-shake ends the kernel instead of hanging it

__global__ void __launch_bounds__(64, 1) k_local_march(MarchArgs a)
{
    extern __shared__ double s_key[];                      // kBandSlots keys ...
    uint32_t* s_xy = (uint32_t*)(s_key + kBandSlots);      // ... and packed (Y << 16 | X) cells
    // warp 0 -> warp 1, one word so that no fence is needed: slot popped [0,14), band head [14,28)
    // and tail [28,42) as they were before the pop, pop number mod 2^22 above
    __shared__ volatile unsigned long long s_pub;
    __shared__ volatile uint32_t s_min_seq;                // scans finished by warp 1
    __shared__ volatile unsigned long long s_mkey;         // its answer: bit pattern of the best key ...
    __shared__ volatile uint32_t s_mslot;                  // ... and its slot
    const LocalView& v = a.v;
    const int lane = threadIdx.x & 31;
    const unsigned full = 0xffffffffu;
    const double inf = DYMU_INF;
    const unsigned long long kInfBits = 0x7FF0000000000000ull;
    const uint32_t w = v.w;
    const uint32_t wg = w / v.r;
    if (threadIdx.x == 0)
    {
        s_pub = 0;
        s_min_seq = 0;
        s_mkey = kInfBits;
        s_mslot = 0xFFFFFFFFu;
    }
    int64_t status = DYMU_LOCAL_OK, end_cell = -1;
    int64_t agent = cell_of(v, a.sx, a.sy);
    int64_t node_end = -1;
    double ex = 0, ey = 0;
    if (agent < 0) status = DYMU_LOCAL_WINDOW_EXCEEDED;
    else if (v.obst[cell_addr(v, agent)]) status = DYMU_LOCAL_START_IN_OBSTACLE;  // L.cpp:610-614
    if (status == DYMU_LOCAL_OK && a.approach == 0)
    {
        node_end = cell_of(v, a.ox, a.oy);  // L.cpp:629
        if (node_end < 0) status = DYMU_LOCAL_WINDOW_EXCEEDED;
        else if (v.obst[cell_addr(v, node_end)]) status = DYMU_LOCAL_END_IN_OBSTACLE;
        else world_pose(v, node_end, ex, ey);
    }
    // the per-axis tables (both warps)
    int32_t* const node_x = a.axis_node;
    int32_t* const node_y = a.axis_node + wg;
    double* const d2_x = a.axis_d2;
    double* const d2_y = a.axis_d2 + w;
    if (status == DYMU_LOCAL_OK)
    {
        for (uint32_t q = threadIdx.x; q < wg; q += 64)
        {
            node_x[q] = nearest_node_axis(v.gres, (double)(v.gx0 + q), v.nx);
            node_y[q] = nearest_node_axis(v.gres, (double)(v.gy0 + q), v.ny);
        }
        if (a.approach == 0)
            for (uint32_t q = threadIdx.x; q < w; q += 64)
            {
                const double dx = world_axis(v, v.gx0, q) - ex, dy = world_axis(v, v.gy0, q) - ey;
                d2_x[q] = dx * dx;
                d2_y[q] = dy * dy;
            }
    }
    __syncthreads();
    if (threadIdx.x >= 32)
    {
        // ---- warp 1: best of the rest for every announced pop
        for (uint32_t k = 1;; ++k)
        {
            unsigned long long pub;
            int spins = 0;
            do pub = s_pub;
            while (pub != kMarchExit && (uint32_t)(pub >> 42) != (k & 0x3FFFFFu) && ++spins < kMarchSpinLimit);
            if (pub == kMarchExit || (uint32_t)(pub >> 42) != (k & 0x3FFFFFu)) return;
            const uint32_t bp = (uint32_t)pub & 0x3FFFu, head = (uint32_t)(pub >> 14) & 0x3FFFu,
                           tail = (uint32_t)(pub >> 28) & 0x3FFFu;
            unsigned long long best = kInfBits;
            uint32_t bslot = 0xFFFFFFFFu;
#pragma unroll 4
            for (uint32_t q = head + lane; q < tail; q += 32)
            {
                const unsigned long long kb = (unsigned long long)__double_as_longlong(s_key[q]);
                if (kb < best && q != bp)
                {
                    best = kb;
                    bslot = q;
                }
            }
            const uint32_t hi = (uint32_t)(best >> 32), lo = (uint32_t)best;
            const uint32_t mhi = __reduce_min_sync(full, hi);
            const uint32_t mlo = __reduce_min_sync(full, hi == mhi ? lo : 0xFFFFFFFFu);
            const uint32_t ms = __reduce_min_sync(full, (hi == mhi && lo == mlo) ? bslot : 0xFFFFFFFFu);
            if (lane == 0)
            {
                s_mkey = ((unsigned long long)mhi << 32) | mlo;
                s_mslot = mhi >= 0x7FF00000u ? 0xFFFFFFFFu : ms;
                __threadfence_block();
                s_min_seq = k;
            }
            __syncwarp();
        }
    }
    const int64_t bx = v.gx0 * (int64_t)v.r, by = v.gy0 * (int64_t)v.r;
    // the global map in window coordinates, clamped just outside the window: all the
    // neighbour classification below is 32-bit compares
    const MapBox box = {clamp_box(-bx, w), clamp_box((int64_t)v.nx * v.r - bx, w),
                        clamp_box(-by, w), clamp_box((int64_t)v.ny * v.r - by, w), (int)w};
    // floor(X / r) == umulhi(X, r_magic) for X, r < 2^16 (r == 1 would need 2^32: handled apart)
    const uint32_t r_magic = 0xFFFFFFFFu / v.r + 1;
    const bool r_is_one = v.r == 1;
    // cells whose four neighbours are all inside the window and the map: no classification needed
    const int ix0 = max(box.x0, 0) + 1, iy0 = max(box.y0, 0) + 1;
    const unsigned ixs = (unsigned)max(min(box.x1, (int)w) - 1 - ix0, 0),
                   iys = (unsigned)max(min(box.y1, (int)w) - 1 - iy0, 0);
    uint32_t* pos = a.nb;  // per window cell: slot of the node while it is in the band
    // reset of the previous propagation, L.cpp:589-599
    for (uint32_t q = lane; q < a.prev_prop; q += 32)
    {
        uint32_t c = a.prop[q];
        size_t o = (size_t)(c / w) * v.pitch + c % w;
        v.state[o] = 0;
        v.dev[o] = inf;
        v.ltot[o] = inf;
    }
    __syncwarp();
    uint64_t closed = 0;
    uint32_t head = 0, tail = 0, live = 0, prop_n = 0, nb_peak = 0;
    if (status == DYMU_LOCAL_OK)
    {
        if (lane == 0)
        {
            size_t o = cell_addr(v, agent);
            uint32_t AX = (uint32_t)(agent % w), AY = (uint32_t)(agent / w);
            v.dev[o] = 0;
            v.ltot[o] = local_total_cost(v, agent);
            v.state[o] = 1;
            double key = 0;
            if (a.approach == 0)
            {
                double wx, wy;
                world_xy(v, AX, AY, wx, wy);
                key = key + sqrt((wx - ex) * (wx - ex) + (wy - ey) * (wy - ey));
            }
            s_xy[0] = (AY << 16) | AX;
            s_key[0] = key;
            pos[agent] = 0;
            a.prop[0] = (uint32_t)agent;
        }
        tail = live = prop_n = 1;
        __syncwarp();
    }
    uint64_t pops = 0;
#ifdef DYMU_LOCAL_PROFILE
    long long lm_t[8] = {0, 0, 0, 0, 0, 0, 0, 0}, lm_last = clock64();
#define LM_MARK(k)                    \
    {                                 \
        long long now_ = clock64();   \
        lm_t[k] += now_ - lm_last;    \
        lm_last = now_;               \
    }
#else
#define LM_MARK(k)
#endif
    bool end_ready = false, end_closed = false;
    int64_t end_addr = -1;  // lanes 0..3: the end node's neighbours, lane 4: the end node
    // the band entries the previous pop lowered or created (lanes 0..3): (key bits, slot); before
    // the first pop that is the agent's entry in slot 0
    unsigned long long ev_key = kInfBits;
    uint32_t ev_slot = 0xFFFFFFFFu;
    if (status == DYMU_LOCAL_OK && lane == 0)
    {
        ev_key = (unsigned long long)__double_as_longlong(s_key[0]);
        ev_slot = 0;
    }
    const int ndx = (lane == 2) - (lane == 1), ndy = (lane == 3) - (lane == 0);  // nb4 order, L.cpp:57-65
    bool rescan = false;  // the slots were renumbered: this pop scans the band itself
    auto wait_scan = [&](uint32_t k) -> bool {
        int spins = 0;
        while (s_min_seq < k)
            if (++spins >= kMarchSpinLimit) return false;
        return true;
    };
    while (status == DYMU_LOCAL_OK)
    {
        if (live == 0) { status = DYMU_LOCAL_EXHAUSTED; break; }
        if (++pops > a.max_pops) { status = DYMU_LOCAL_EXHAUSTED; break; }
        // ---- housekeeping: stable compaction of the slot array
        // warp 1's scan for the previous pop has to be finished before its answer is used -- and
        // before the slots may be renumbered under it
        if (!wait_scan((uint32_t)pops - 1)) { status = DYMU_LOCAL_EXHAUSTED; break; }
        if (tail + 4 > kBandSlots || tail - head > live + 64)
        {
            rescan = true;
            uint32_t dst = 0;
            for (uint32_t base = head; base < tail; base += 32)
            {
                uint32_t q = base + lane;
                double k = (q < tail) ? s_key[q] : inf;
                uint32_t xy = (q < tail) ? s_xy[q] : 0;
                bool keep = k < inf;
                unsigned m = __ballot_sync(full, keep);
                __syncwarp();
                if (keep)
                {
                    uint32_t d = dst + __popc(m & ((1u << lane) - 1));
                    s_key[d] = k;
                    s_xy[d] = xy;
                    pos[(xy >> 16) * w + (xy & 0xffffu)] = d;
                }
                dst += __popc(m);
                __syncwarp();
            }
            head = 0;
            tail = dst;
            if (tail + 4 > kBandSlots) { status = DYMU_LOCAL_WINDOW_EXCEEDED; break; }
        }
        LM_MARK(0);
        // ---- minCostLocalNode: strict '<' argmin, earliest position wins (L.cpp:752-805)
        uint32_t bp;
        if (rescan)
        {
            double bk0 = inf;
            uint32_t bp0 = 0xFFFFFFFFu;
#pragma unroll 4
            for (uint32_t q = head + lane; q < tail; q += 32)
            {
                double key = s_key[q];
                if (key < bk0)
                {
                    bk0 = key;
                    bp0 = q;
                }
            }
            // lexicographic (key, slot) minimum over the lanes; keys are non-negative (or +inf
            // for "nothing"), so their bit patterns order like the values
            const unsigned long long kb = (unsigned long long)__double_as_longlong(bk0);
            const uint32_t hi = (uint32_t)(kb >> 32), lo = (uint32_t)kb;
            const uint32_t mhi = __reduce_min_sync(full, hi);
            const uint32_t mlo = __reduce_min_sync(full, hi == mhi ? lo : 0xFFFFFFFFu);
            bp = __reduce_min_sync(full, (hi == mhi && lo == mlo) ? bp0 : 0xFFFFFFFFu);
            rescan = false;
        }
        else
        {
            // best of the rest (warp 1, lane 4 here) against what the previous pop touched (lanes 0..3)
            unsigned long long ck = lane < 4 ? ev_key : kInfBits;
            uint32_t cs = lane < 4 ? ev_slot : 0xFFFFFFFFu;
            if (lane == 4)
            {
                ck = s_mkey;
                cs = s_mslot;
            }
            if (cs == 0xFFFFFFFFu) ck = kInfBits;
            const uint32_t hi = (uint32_t)(ck >> 32), lo = (uint32_t)ck;
            const uint32_t mhi = __reduce_min_sync(full, hi);
            const uint32_t mlo = __reduce_min_sync(full, hi == mhi ? lo : 0xFFFFFFFFu);
            bp = __reduce_min_sync(full, (hi == mhi && lo == mlo) ? cs : 0xFFFFFFFFu);
            if (mhi >= 0x7FF00000u) bp = 0xFFFFFFFFu;
        }
        if (bp == 0xFFFFFFFFu) { status = DYMU_LOCAL_EXHAUSTED; break; }
        if (lane == 0)
            s_pub = (unsigned long long)bp | ((unsigned long long)head << 14) | ((unsigned long long)tail << 28)
                    | ((unsigned long long)((uint32_t)pops & 0x3FFFFFu) << 42);
        const uint32_t pxy = s_xy[bp];
        const int X = (int)(pxy & 0xffffu), Y = (int)(pxy >> 16);
        const size_t oX = (size_t)Y * v.pitch + X;
        __syncwarp();
        // ---- vector::erase(begin + bp)
        if (lane == 0)
        {
            s_key[bp] = inf;
            v.state[oX] = 1;  // CLOSED, L.cpp:653
        }
        live--;
        closed++;
        __syncwarp();
        if (bp == head)
        {
            uint32_t h = head + 1;
            while (h < tail)
            {
                bool lv = (h + lane < tail) && (s_key[h + lane] < inf);
                unsigned m = __ballot_sync(full, lv);
                if (m) { h += __ffs(m) - 1; break; }
                h += 32;
            }
            head = min(h, tail);
        }
        LM_MARK(1);
        // ---- the four neighbours on lanes 0..3 (independent: no target is another's input).
        // Every value the update may need is requested up front so that a pop costs one
        // memory round trip, not a chain of them.
        int nX = X, nY = Y;
        size_t o = 0;
        uint32_t lin = 0;
        bool is_end_candidate = false, is_new = false, lowered = false;
        double newkey = 0;
        ev_key = kInfBits;
        ev_slot = 0xFFFFFFFFu;
        if (lane < 5 && oX == (size_t)end_addr) end_closed = true;
        if (lane < 4)
        {
            nX += ndx;
            nY += ndy;
            int cls = 0, c0 = 0, c1 = 0, c2 = 0, c3 = 0;
            if ((unsigned)(nX - ix0) >= ixs || (unsigned)(nY - iy0) >= iys)
            {
                cls = box_class(box, nX, nY);
                c0 = box_class(box, nX, nY - 1);
                c1 = box_class(box, nX - 1, nY);
                c2 = box_class(box, nX + 1, nY);
                c3 = box_class(box, nX, nY + 1);
            }
            if (cls == -2) status = DYMU_LOCAL_WINDOW_EXCEEDED;
            if (cls == 0)
            {
                o = (size_t)((uint32_t)nY * v.pitch + (uint32_t)nX);
                lin = (uint32_t)nY * w + (uint32_t)nX;
                const uint8_t st = v.state[o], ob = v.obst[o];
                const double d0 = (c0 == 0) ? v.dev[o - v.pitch] : inf, d1 = (c1 == 0) ? v.dev[o - 1] : inf,
                             d2 = (c2 == 0) ? v.dev[o + 1] : inf, d3 = (c3 == 0) ? v.dev[o + v.pitch] : inf;
                const double R = v.risk[o], cur = v.dev[o], lt0 = v.ltot[o], ltc = a.ltot_cache[o];
                const uint32_t slot = pos[lin];
                double h2 = 0;  // CONSERVATIVE: squared distance to the end node, L.cpp:735-741
                if (a.approach == 0) h2 = d2_x[nX] + d2_y[nY];
                LM_MARK(4);
                // L.cpp:658-663: looking at a neighbour under a different parent subdivides it
                const uint32_t PX = r_is_one ? (uint32_t)X : __umulhi((uint32_t)X, r_magic),
                               PY = r_is_one ? (uint32_t)Y : __umulhi((uint32_t)Y, r_magic),
                               QX = r_is_one ? (uint32_t)nX : __umulhi((uint32_t)nX, r_magic),
                               QY = r_is_one ? (uint32_t)nY : __umulhi((uint32_t)nY, r_magic);
                if (QX != PX || QY != PY)
                {
                    const int32_t gi = node_x[QX], gj = node_y[QY], pi = node_x[PX], pj = node_y[PY];
                    if ((gi | gj | pi | pj) >= 0 && (gi != pi || gj != pj))
                    {
                        int64_t ex_ = gi - v.gx0, ey_ = gj - v.gy0;
                        if (ex_ >= 0 && ey_ >= 0 && ex_ < wg && ey_ < wg) a.entered[ey_ * wg + ex_] = 1;
                    }
                }
                LM_MARK(5);
                if ((st == 0) && (!ob))  // L.cpp:664-665
                {
                    LM_MARK(6);
                    // propagateLocalNode, L.cpp:700-750
                    if (c0 == -2 || c1 == -2 || c2 == -2 || c3 == -2) status = DYMU_LOCAL_WINDOW_EXCEEDED;
                    else
                    {
                        // neighbour pair rule, L.cpp:705-717 (a missing neighbour reads as +inf)
                        double Ty = (c0 == 0 && c3 == 0) ? fmin(d3, d0) : ((c0 != 0) ? d3 : d0);
                        double Tx = (c1 == 0 && c2 == 0) ? fmin(d2, d1) : ((c1 != 0) ? d2 : d1);
                        double lt = lt0;
                        if (lt == inf) { lt = ltc; v.ltot[o] = lt; }
                        double C = v.lres * (a.risk_ratio * R + 1);
                        double Tn = dymu_eikonal(Tx, Ty, C);
                        if (Tn < cur)
                        {
                            LM_MARK(7);
                            is_new = (cur == inf);
                            lowered = true;
                            v.dev[o] = Tn;
                            newkey = Tn;
                            if (a.approach == 0) newkey = newkey + sqrt(h2);
                            if (!is_new)
                            {
                                s_key[slot] = newkey;
                                ev_slot = slot;
                            }
                            ev_key = (unsigned long long)__double_as_longlong(newkey);
                        }
                        is_end_candidate = (lt < a.t_overtake) && (R == 0);  // L.cpp:668-671
                    }
                }
            }
        }
        status = __reduce_max_sync(full, (int)status);
        LM_MARK(2);
        if (status != DYMU_LOCAL_OK) break;
        // push_back in nb4 order, L.cpp:742-747
        unsigned newmask = __ballot_sync(full, is_new);
        uint32_t added = __popc(newmask);
        if (prop_n + added >= a.cap) { status = DYMU_LOCAL_WINDOW_EXCEEDED; break; }
        if (is_new)
        {
            uint32_t off = __popc(newmask & ((1u << lane) - 1));
            s_xy[tail + off] = ((uint32_t)nY << 16) | (uint32_t)nX;
            s_key[tail + off] = newkey;
            pos[lin] = tail + off;
            a.prop[prop_n + off] = lin;
            ev_slot = tail + off;
        }
        tail += added;
        live += added;
        prop_n += added;
        nb_peak = max(nb_peak, live);
        if (node_end < 0)
        {
            unsigned cm = __ballot_sync(full, is_end_candidate);
            if (cm)
            {
                int src = __ffs(cm) - 1;
                node_end = (int64_t)__shfl_sync(full, lin, src);
            }
        }
        __syncwarp();
        LM_MARK(3);
        // ---- end test, L.cpp:674-684: the end node and its four neighbours are CLOSED.
        // Their state is read once when the end node becomes known and then followed in
        // registers (a node is CLOSED exactly when it is popped).
        if (node_end >= 0)
        {
            if (!end_ready)
            {
                if (lane < 5)
                {
                    int64_t c = (lane == 4) ? node_end : lnb4(v, node_end, lane);
                    end_addr = (c >= 0) ? (int64_t)cell_addr(v, c) : -1;
                    end_closed = (end_addr >= 0) && (v.state[end_addr] == 1);
                }
                end_ready = true;
            }
            if (__all_sync(full, lane >= 5 || end_closed))
            {
                end_cell = node_end;
                break;
            }
        }
    }
    if (lane == 0)
    {
        s_pub = kMarchExit;  // releases warp 1
        a.result[0] = (status == DYMU_LOCAL_OK) ? end_cell : -1;
        a.result[1] = status;
        a.result[2] = (int64_t)closed;
        a.result[3] = prop_n;
        a.result[4] = nb_peak;
#ifdef DYMU_LOCAL_PROFILE
        // cycles: [5] end test + housekeeping, [6] argmin + erase, [7] neighbours, [8] push
        for (int k = 0; k < 8; ++k) a.result[5 + k] = lm_t[k];
#endif
    }
}

// ---------------------------------------------------------------------------------
// local path extraction
// ---------------------------------------------------------------------------------
struct LPathArgs
{
    LocalView v;
    int64_t end_cell;
    double sx, sy;         // wayp_start
    double off_x, off_y;   // global_offset (subtracted again in L.cpp:890-891)
    double* out;           // 6 doubles per waypoint
    uint32_t cap;
    uint32_t* result;      // [0] n [1] status
};

__device__ __forceinline__ double lgrad_axis(const LocalView& v, int64_t c, int64_t lo, int64_t hi)
{
    const double inf = DYMU_INF;
    const double* F = v.dev;
    bool hl = lo >= 0, hh = hi >= 0;
    double f = F[cell_addr(v, c)];
    double flo = hl ? F[cell_addr(v, lo)] : 0, fhi = hh ? F[cell_addr(v, hi)] : 0;
    if ((!hl && !hh) || (hl && hh && flo == inf && fhi == inf)) return 0;
    if (!hl || flo == inf)
    {
        if (!hh) return 0;
        return fhi - f;
    }
    if (!hh || fhi == inf) return f - flo;
    return (fhi - flo) * 0.5;
}

// gradientNode(localNode*), L.cpp:979-1023: no guard for the zero vector (0/0 -> NaN)
__device__ __forceinline__ void lgrad_node(const LocalView& v, int64_t c, double& dnx, double& dny)
{
    if (c < 0)
    {
        dnx = dny = __longlong_as_double(0x7FF8000000000000LL);
        return;
    }
    double dx = lgrad_axis(v, c, lnb4(v, c, 1), lnb4(v, c, 2));
    double dy = lgrad_axis(v, c, lnb4(v, c, 0), lnb4(v, c, 3));
    double n = sqrt(dx * dx + dy * dy);
    dnx = dx / n;
    dny = dy / n;
}

__device__ __forceinline__ int64_t nn(const LocalView& v, int64_t c, int d)
{
    int64_t r = lnb4(v, c, d);
    return r < 0 ? -1 : r;
}

// computeLocalWaypointGDM, L.cpp:877-977.  w = {x, y, z}; d = gradient used
__device__ bool local_gdm(const LPathArgs& a, int lane, double* w, double tau, double& dCx,
                          double& dCy)
{
    const LocalView& v = a.v;
    int64_t L = cell_of(v, w[0], w[1]);
    // elevation (swapped corners, L.cpp:900-905) at the global cell of the doubly offset position
    double gXp = w[0] - a.off_x, gYp = w[1] - a.off_y;
    double fx = gXp / v.gres, fy = gYp / v.gres;
    if (fx >= 0 && fy >= 0 && fx < (double)(v.nx - 1) && fy < (double)(v.ny - 1))
    {
        uint32_t cx = (uint32_t)fx, cy = (uint32_t)fy;
        double dX = gXp - (double)cx, dY = gYp - (double)cy;
        const double* e = v.elev + (size_t)cy * v.gpitch + cx;
        w[2] = dymu_interp(dX, dY, e[0], e[1], e[v.gpitch], e[v.gpitch + 1]);
    }
    if (L < 0)
    {
        dCx = dCy = __longlong_as_double(0x7FF8000000000000LL);
        return false;
    }
    double lwx, lwy, aa, bb;
    world_pose(v, L, lwx, lwy);
    int64_t n00, n10, n01, n11;
    if (lwx < w[0])
    {
        if (lwy < w[1])
        {
            n00 = L; n10 = nn(v, L, 2); n01 = nn(v, L, 3); n11 = nn(v, nn(v, L, 2), 3);
            aa = (w[0] - lwx) / v.lres; bb = (w[1] - lwy) / v.lres;
        }
        else
        {
            n00 = nn(v, L, 0); n10 = nn(v, L, 2); n01 = L; n11 = nn(v, nn(v, L, 0), 2);
            aa = (w[0] - lwx) / v.lres; bb = 1 + (w[1] - lwy) / v.lres;
        }
    }
    else
    {
        if (lwy < w[1])
        {
            n00 = nn(v, L, 1); n10 = L; n01 = nn(v, L, 3); n11 = nn(v, nn(v, L, 3), 1);
            aa = 1 + (w[0] - lwx) / v.lres; bb = (w[1] - lwy) / v.lres;
        }
        else
        {
            n00 = nn(v, nn(v, L, 1), 0); n10 = nn(v, L, 0); n01 = nn(v, L, 1); n11 = L;
            aa = 1 + (w[0] - lwx) / v.lres; bb = 1 + (w[1] - lwy) / v.lres;
        }
    }
    // the four corner gradients on lanes 0..3
    int c = lane & 3;
    int64_t mine = (c == 0) ? n00 : (c == 1) ? n10 : (c == 2) ? n01 : n11;
    double gxc, gyc;
    lgrad_node(v, mine, gxc, gyc);
    const unsigned full = 0xffffffffu;
    double gx00 = __shfl_sync(full, gxc, 0), gx10 = __shfl_sync(full, gxc, 1);
    double gx01 = __shfl_sync(full, gxc, 2), gx11 = __shfl_sync(full, gxc, 3);
    double gy00 = __shfl_sync(full, gyc, 0), gy10 = __shfl_sync(full, gyc, 1);
    double gy01 = __shfl_sync(full, gyc, 2), gy11 = __shfl_sync(full, gyc, 3);
    dCx = dymu_interp(aa, bb, gx00, gx01, gx10, gx11);
    dCy = dymu_interp(aa, bb, gy00, gy01, gy10, gy11);
    if (isnan(dCx) || isnan(dCy)) return false;
    if (sqrt(dCx * dCx + dCy * dCy) < 0.001 * tau * v.lres) return false;
    w[0] = w[0] - tau * dCx;
    w[1] = w[1] - tau * dCy;
    return true;
}

// getLocalPath, L.cpp:807-849
__global__ void __launch_bounds__(32, 1) k_local_path(LPathArgs a)
{
    const LocalView& v = a.v;
    const int lane = threadIdx.x;
    uint32_t n = 0, status = DYMU_PATH_OK;
    double w[3], dCx, dCy;
    global_pose(v, a.end_cell, w[0], w[1]);
    w[2] = 0.0;
    double tau = 0.5 * v.lres;
    // the two most recently inserted waypoints (trajectory[0], trajectory[1])
    double f0x = 0, f0y = 0, f1y = 0;
    auto push = [&](double kind, double dx, double dy) -> bool {
        if (n >= a.cap) return false;
        if (lane == 0)
        {
            double* o = a.out + (size_t)6 * n;
            o[0] = w[0]; o[1] = w[1]; o[2] = w[2]; o[3] = dx; o[4] = dy; o[5] = kind;
        }
        if (n > 0) f1y = f0y;
        f0x = w[0];
        f0y = w[1];
        n++;
        return true;
    };
    bool valid = local_gdm(a, lane, w, tau * v.lres, dCx, dCy);
    // an invalid first step leaves wPos unchanged with the end node's heading (L.cpp:815-820)
    push(valid ? 0.0 : 2.0, dCx, dCy);
    while (sqrt((f0x - a.sx) * (f0x - a.sx) + (f0y - a.sy) * (f0y - a.sy)) > 1.5 * v.lres)
    {
        valid = local_gdm(a, lane, w, tau, dCx, dCy);
        if (n > 1)
        {
            // L.cpp:830-833 mixes trajectory[0].x with trajectory[1].y; with a single element
            // the reference reads out of bounds (quirk 6) and the test is treated as not taken
            double ddx = w[0] - f0x, ddy = w[1] - f1y;
            if (sqrt(ddx * ddx + ddy * ddy) < 0.01 * tau * v.lres) valid = false;
        }
        if (valid)
        {
            if (!push(0.0, dCx, dCy)) { status = DYMU_PATH_CAPACITY; break; }
        }
        else
        {
            // computeLocalWaypointDijkstra, L.cpp:851-869, from the node under trajectory[0]
            int64_t L = cell_of(v, f0x, f0y);
            double t = DYMU_INF, newX = 0, newY = 0, lx = 0, ly = 0;
            if (L >= 0)
            {
                for (int d = 0; d < 4; ++d)
                {
                    int64_t nb = lnb4(v, L, d);
                    if (nb >= 0)
                    {
                        double dv = v.dev[cell_addr(v, nb)];
                        if (dv < t) { t = dv; world_pose(v, nb, newX, newY); }
                    }
                }
                world_pose(v, L, lx, ly);
            }
            if (!(t < DYMU_INF)) { status = DYMU_PATH_STALLED; break; }
            w[0] = newX; w[1] = newY; w[2] = 0.0;
            if (!push(1.0, newX - lx, newY - ly)) { status = DYMU_PATH_CAPACITY; break; }
        }
    }
    if (lane == 0)
    {
        a.result[0] = n;
        a.result[1] = status;
    }
}

__global__ void k_sample_risk(LocalView v, const double* xy, uint32_t n, double* out)
{
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    int64_t c = cell_of(v, xy[2 * k], xy[2 * k + 1]);
    out[k] = (c >= 0) ? v.risk[cell_addr(v, c)] : 0.0;
}

__global__ void k_cell_of(LocalView v, double x, double y, int64_t* out) { *out = cell_of(v, x, y); }

LocalView make_view(const dymu_ctx* ctx)
{
    const dymu_local& l = ctx->loc;
    LocalView v;
    v.risk = l.risk; v.dev = l.dev; v.ltot = l.ltot; v.obst = l.obst; v.state = l.state;
    v.w = l.w; v.pitch = l.pitch; v.r = l.r; v.gx0 = l.gx0; v.gy0 = l.gy0;
    v.nx = ctx->nx; v.ny = ctx->ny; v.gres = ctx->gres; v.lres = ctx->lres;
    v.T = ctx->T; v.elev = ctx->elev; v.gobst = ctx->obst; v.gpitch = ctx->pitch;
    return v;
}

}  // namespace

static dymu_local* extra_of(dymu_ctx* ctx) { return &ctx->loc; }

static void local_release(dymu_local& l);
void dymu_internal_local_free(dymu_ctx* ctx) { local_release(ctx->loc); }

static int local_clear(dymu_ctx* ctx)
{
    dymu_local& l = ctx->loc;
    size_t n = (size_t)l.pitch * l.rows;
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(l.risk, 0, n * sizeof(double), ctx->stream));
    DYMU_TRY(dymu_internal_fill(ctx, l.dev, 1.0 / 0.0, n));
    DYMU_TRY(dymu_internal_fill(ctx, l.ltot, 1.0 / 0.0, n));
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(l.obst, 0, n, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(l.state, 0, n, ctx->stream));
    dymu_local* e = extra_of(ctx);
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(e->entered, 0, (size_t)l.wg * l.wg, ctx->stream));
    e->prop_count = 0;
    return DYMU_OK;
}

// Allocates the planes of a wg x wg window into `l` (which must not own memory) and clears them.
static int local_alloc(dymu_ctx* ctx, dymu_local& l, uint32_t wg)
{
    memset(&l, 0, sizeof(l));
    l.wg = wg;
    l.r = (uint32_t)(ctx->gres / ctx->lres);  // res_ratio, G.cpp:49
    if (l.r < 1) DYMU_FAIL(ctx, DYMU_ERR_ARG, "local_res must not exceed global_res");
    if ((uint64_t)wg * l.r > 65535u) DYMU_FAIL(ctx, DYMU_ERR_ARG, "local window of %u nodes is too large", wg);
    l.w = wg * l.r;
    l.pitch = dymu_div_up(l.w, kTile) * kTile;
    l.rows = l.pitch;
    size_t n = (size_t)l.pitch * l.rows;
    double** f64[] = {&l.risk, &l.dev, &l.ltot, &l.crisk};
    for (double** p : f64) DYMU_CUDA_TRY(ctx, cudaMalloc((void**)p, n * sizeof(double)));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&l.obst, n));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&l.state, n));
    l.nb_cap = l.w * l.w;
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&l.nb_idx, (size_t)l.nb_cap * sizeof(uint32_t)));
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(l.nb_idx, 0, (size_t)l.nb_cap * sizeof(uint32_t), ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&l.first, (size_t)l.w * l.w * sizeof(uint32_t)));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&l.prop, (size_t)l.nb_cap * sizeof(uint32_t)));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&l.entered, (size_t)wg * wg));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&l.axis_d2, (size_t)2 * l.w * sizeof(double)));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&l.axis_node, (size_t)2 * wg * sizeof(int32_t)));
    uint32_t nt = l.pitch / kTile;
    DYMU_TRY(dymu_internal_fim_alloc(ctx, &l.work, (size_t)nt * nt));
    l.allocated = true;
    return DYMU_OK;
}

static void local_release(dymu_local& l)
{
    if (!l.allocated) return;
    dymu_internal_fim_free(&l.work);
    void* ptrs[] = {l.risk, l.dev, l.ltot, l.crisk, l.obst, l.state, l.nb_idx, l.first, l.prop, l.entered,
                    l.axis_d2, l.axis_node};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    memset(&l, 0, sizeof(l));
}

// deviation / total cost / state of every window cell back to "never propagated" (what the
// reference's per-propagation reset of local_propagated_nodes, L.cpp:589-599, leaves behind)
static int local_reset_wave(dymu_ctx* ctx)
{
    dymu_local& l = ctx->loc;
    size_t n = (size_t)l.pitch * l.rows;
    DYMU_TRY(dymu_internal_fill(ctx, l.dev, 1.0 / 0.0, n));
    DYMU_TRY(dymu_internal_fill(ctx, l.ltot, 1.0 / 0.0, n));
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(l.state, 0, n, ctx->stream));
    l.prop_count = 0;
    return DYMU_OK;
}

extern "C" {

int dymu_local_create(dymu_ctx* ctx, uint32_t wg)
{
    DYMU_GUARD(ctx);
    CallTrace call_trace(__func__);
    if (!ctx || wg < 3) return DYMU_ERR_ARG;
    dymu_internal_local_free(ctx);
    DYMU_TRY(local_alloc(ctx, ctx->loc, wg));
    ctx->loc.gx0 = ctx->loc.gy0 = 0;
    return local_clear(ctx);
}

int dymu_local_anchor(dymu_ctx* ctx, int64_t gx0, int64_t gy0)
{
    DYMU_GUARD(ctx);
    CallTrace call_trace(__func__);
    if (!ctx || !ctx->loc.allocated) return DYMU_ERR_STATE;
    ctx->loc.gx0 = gx0;
    ctx->loc.gy0 = gy0;
    return local_clear(ctx);
}

int dymu_local_reshape(dymu_ctx* ctx, uint32_t wg, int64_t gx0, int64_t gy0)
{
    DYMU_GUARD(ctx);
    CallTrace call_trace(__func__);
    if (!ctx || wg < 3) return DYMU_ERR_ARG;
    if (!ctx->loc.allocated)
    {
        DYMU_TRY(local_alloc(ctx, ctx->loc, wg));
        ctx->loc.gx0 = gx0;
        ctx->loc.gy0 = gy0;
        return local_clear(ctx);
    }
    dymu_local old = ctx->loc;  // keeps the device pointers of the current window
    dymu_local fresh;
    int rc = local_alloc(ctx, fresh, wg);
    if (rc != DYMU_OK)
    {
        local_release(fresh);
        return rc;
    }
    fresh.gx0 = gx0;
    fresh.gy0 = gy0;
    ctx->loc = fresh;
    rc = local_clear(ctx);
    // the persistent local-node fields -- isObstacle and risk (the reference never forgets a
    // local node, L.cpp:150-156 and the empty destructor G.cpp:36) -- move with the overlap
    const int64_t r = old.r;
    const int64_t ox0 = old.gx0 * r, oy0 = old.gy0 * r, nx0 = gx0 * r, ny0 = gy0 * r;
    const int64_t x0 = std::max(ox0, nx0), y0 = std::max(oy0, ny0);
    const int64_t x1 = std::min(ox0 + (int64_t)old.w, nx0 + (int64_t)fresh.w);
    const int64_t y1 = std::min(oy0 + (int64_t)old.w, ny0 + (int64_t)fresh.w);
    if (rc == DYMU_OK && x1 > x0 && y1 > y0)
    {
        const size_t so = (size_t)(y0 - oy0) * old.pitch + (size_t)(x0 - ox0);
        const size_t dn = (size_t)(y0 - ny0) * fresh.pitch + (size_t)(x0 - nx0);
        const size_t cw = (size_t)(x1 - x0), ch = (size_t)(y1 - y0);
        cudaError_t e1 = cudaMemcpy2DAsync(fresh.risk + dn, fresh.pitch * sizeof(double), old.risk + so,
                                           old.pitch * sizeof(double), cw * sizeof(double), ch,
                                           cudaMemcpyDeviceToDevice, ctx->stream);
        cudaError_t e2 = cudaMemcpy2DAsync(fresh.obst + dn, fresh.pitch, old.obst + so, old.pitch, cw, ch,
                                           cudaMemcpyDeviceToDevice, ctx->stream);
        if (e1 != cudaSuccess || e2 != cudaSuccess)
        {
            snprintf(ctx->err, sizeof(ctx->err), "local window reshape: %s",
                     cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
            rc = DYMU_ERR_CUDA;
        }
    }
    cudaStreamSynchronize(ctx->stream);
    local_release(old);
    return rc;
}

int dymu_local_info(const dymu_ctx* ctx, int64_t* gx0, int64_t* gy0, uint32_t* wg, uint32_t* r)
{
    CallTrace call_trace(__func__);
    if (!ctx || !ctx->loc.allocated) return DYMU_ERR_STATE;
    if (gx0) *gx0 = ctx->loc.gx0;
    if (gy0) *gy0 = ctx->loc.gy0;
    if (wg) *wg = ctx->loc.wg;
    if (r) *r = ctx->loc.r;
    return DYMU_OK;
}

static double* lplane(dymu_ctx* ctx, int p)
{
    switch (p)
    {
        case DYMU_LPLANE_RISK: return ctx->loc.risk;
        case DYMU_LPLANE_DEVIATION: return ctx->loc.dev;
        case DYMU_LPLANE_TOTAL_COST: return ctx->loc.ltot;
        default: return nullptr;
    }
}

int dymu_local_read_rect(dymu_ctx* ctx, int lplane_id, uint32_t x0, uint32_t y0, uint32_t w,
                         uint32_t h, double* host)
{
    DYMU_GUARD(ctx);
    CallTrace call_trace(__func__);
    if (!ctx || !ctx->loc.allocated || !host) return DYMU_ERR_ARG;
    const dymu_local& l = ctx->loc;
    double* d = lplane(ctx, lplane_id);
    if (!d || w == 0 || h == 0 || (uint64_t)x0 + w > l.w || (uint64_t)y0 + h > l.w) return DYMU_ERR_ARG;
    DYMU_CUDA_TRY(ctx, cudaMemcpy2DAsync(host, w * sizeof(double), d + (size_t)y0 * l.pitch + x0,
                                         l.pitch * sizeof(double), w * sizeof(double), h,
                                         cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DYMU_OK;
}

int dymu_local_read_rect_u8(dymu_ctx* ctx, int lplane_id, uint32_t x0, uint32_t y0, uint32_t w,
                            uint32_t h, uint8_t* host)
{
    DYMU_GUARD(ctx);
    CallTrace call_trace(__func__);
    if (!ctx || !ctx->loc.allocated || !host) return DYMU_ERR_ARG;
    const dymu_local& l = ctx->loc;
    uint8_t* d = lplane_id == DYMU_LPLANE_U8_OBSTACLE ? l.obst
                 : lplane_id == DYMU_LPLANE_U8_STATE  ? l.state : nullptr;
    if (!d || w == 0 || h == 0 || (uint64_t)x0 + w > l.w || (uint64_t)y0 + h > l.w) return DYMU_ERR_ARG;
    DYMU_CUDA_TRY(ctx, cudaMemcpy2DAsync(host, w, d + (size_t)y0 * l.pitch + x0, l.pitch, w, h,
                                         cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DYMU_OK;
}

int dymu_local_ingest(dymu_ctx* ctx, const uint8_t* image, uint32_t w, uint32_t h,
                      uint32_t row_size, uint32_t pixel_size, double res, double rover_x,
                      double rover_y, uint32_t* new_cells, uint32_t cap, uint32_t* n_new)
{
    DYMU_GUARD(ctx);
    CallTrace call_trace(__func__);
    if (!ctx || !ctx->loc.allocated || !image || !new_cells || !n_new || w == 0 || h == 0
        || row_size < w * pixel_size || pixel_size == 0)
        return DYMU_ERR_ARG;
    const dymu_local& l = ctx->loc;
    dymu_local* e = extra_of(ctx);
    size_t img_bytes = (size_t)row_size * h, npx = (size_t)w * h;
    size_t dev_need = img_bytes + 16 + npx * 4 + 64;
    DYMU_TRY(dymu_internal_scratch(ctx, dev_need, (img_bytes > npx * 4 ? img_bytes : npx * 4) + 64));
    uint8_t* d_img = (uint8_t*)ctx->d_scratch;
    size_t off = (img_bytes + 15) & ~(size_t)15;
    uint32_t* d_flags = (uint32_t*)((char*)ctx->d_scratch + off);
    uint32_t* d_winner = d_flags + 4;
    memcpy(ctx->h_pinned, image, img_bytes);
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(d_img, ctx->h_pinned, img_bytes, cudaMemcpyHostToDevice,
                                       ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(d_flags, 0, 16, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(e->first, 0xFF, (size_t)l.w * l.w * 4, ctx->stream));
    IngestArgs a;
    a.v = make_view(ctx);
    a.image = d_img; a.w = w; a.h = h; a.row_size = row_size; a.pixel_size = pixel_size;
    a.res = res; a.rover_x = rover_x; a.rover_y = rover_y;
    a.first = e->first; a.winner = d_winner; a.flags = d_flags;
    int grid = (int)dymu_div_up((uint32_t)npx, 128);
    k_ingest_claim<<<grid, 128, 0, ctx->stream>>>(a);
    k_ingest_mark<<<grid, 128, 0, ctx->stream>>>(a);
    k_ingest_commit<<<grid, 128, 0, ctx->stream>>>(a);
    ctx->launches += 3;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    uint32_t h_flags[4];
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(h_flags, d_flags, 16, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_pinned, d_winner, npx * 4, cudaMemcpyDeviceToHost,
                                       ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (h_flags[0]) DYMU_FAIL(ctx, DYMU_ERR_CAPACITY, "frame footprint leaves the local window");
    const uint32_t* win = (const uint32_t*)ctx->h_pinned;
    uint32_t n = 0;
    for (size_t p = 0; p < npx; ++p)  // raster order, as the reference visits pixels
        if (win[p] != kNoCell)
        {
            if (n < cap) new_cells[n] = win[p];
            n++;
        }
    *n_new = n;
    if (n > cap) DYMU_FAIL(ctx, DYMU_ERR_CAPACITY, "new obstacle list needs %u entries", n);
    return DYMU_OK;
}

int dymu_local_blocking(dymu_ctx* ctx, const uint32_t* cells, uint32_t n_cells,
                        const double* path_xy, uint32_t n_path, double risk_distance,
                        uint32_t* min_index, uint32_t* max_index, int* blocked)
{
    DYMU_GUARD(ctx);
    CallTrace call_trace(__func__);
    if (!ctx || !ctx->loc.allocated || !min_index || !max_index || !blocked) return DYMU_ERR_ARG;
    *blocked = 0;
    if (n_cells == 0 || n_path == 0) return DYMU_OK;
    size_t need = (size_t)n_cells * 4 + (size_t)n_path * 16 + 64;
    DYMU_TRY(dymu_internal_scratch(ctx, need, need));
    char* hp = (char*)ctx->h_pinned;
    uint32_t* h_out = (uint32_t*)hp;
    h_out[0] = *min_index; h_out[1] = *max_index; h_out[2] = 0; h_out[3] = 0;
    memcpy(hp + 16, path_xy, (size_t)n_path * 16);
    memcpy(hp + 16 + (size_t)n_path * 16, cells, (size_t)n_cells * 4);
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_scratch, hp, 16 + (size_t)n_path * 16 + (size_t)n_cells * 4,
                                       cudaMemcpyHostToDevice, ctx->stream));
    char* dp = (char*)ctx->d_scratch;
    k_blocking<<<dymu_div_up(n_cells, 4), 128, 0, ctx->stream>>>(
        make_view(ctx), (const uint32_t*)(dp + 16 + (size_t)n_path * 16), n_cells,
        (const double*)(dp + 16), n_path, risk_distance, (uint32_t*)dp);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(h_out, dp, 16, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *min_index = h_out[0];
    *max_index = h_out[1];
    *blocked = (int)h_out[2];
    return DYMU_OK;
}

int dymu_local_expand_risk(dymu_ctx* ctx, double risk_distance, dymu_solve_stats* stats)
{
    DYMU_GUARD(ctx);
    CallTrace call_trace(__func__);
    if (!ctx || !ctx->loc.allocated || !(risk_distance > 0)) return DYMU_ERR_ARG;
    dymu_local& l = ctx->loc;
    size_t n = (size_t)l.pitch * l.rows;
    int grid = (int)((n + 255) / 256);
    if (grid > ctx->sm_count * 16) grid = ctx->sm_count * 16;
    k_risk_cplane<<<grid, 256, 0, ctx->stream>>>(l.obst, l.crisk, ctx->lres / risk_distance, l.pitch,
                                                 l.rows, l.w);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    uint32_t nt = l.pitch / kTile;
    DYMU_TRY(dymu_internal_fim_seed_all(ctx, &l.work, nt * nt));
    dymu_fim_launch L;
    L.T = l.risk; L.slot_stride = n; L.C = l.crisk; L.pitch = l.pitch; L.rows = l.rows;
    L.ntx = nt; L.nty = nt; L.nprob = 1; L.mode = 1; L.work = &l.work;
    L.band = 1.0 / 0.0;  // small window: plain FIM
    DYMU_TRY(dymu_internal_fim_run(ctx, L, stats));
    k_mark_entered_risk<<<grid, 256, 0, ctx->stream>>>(make_view(ctx), l.entered);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    return DYMU_OK;
}

int dymu_local_propagate(dymu_ctx* ctx, int approach, double start_x, double start_y,
                         double overtake_x, double overtake_y, double t_overtake,
                         double risk_ratio, int64_t* end_cell, uint32_t* status,
                         uint64_t* n_closed)
{
    DYMU_GUARD(ctx);
    CallTrace call_trace(__func__);
    if (!ctx || !ctx->loc.allocated || !end_cell || !status) return DYMU_ERR_ARG;
    dymu_local& l = ctx->loc;
    dymu_local* e = extra_of(ctx);
    DYMU_TRY(dymu_internal_scratch(ctx, 256, 256));
    MarchArgs a;
    a.v = make_view(ctx);
    a.approach = approach;
    a.sx = start_x; a.sy = start_y; a.ox = overtake_x; a.oy = overtake_y;
    a.t_overtake = t_overtake; a.risk_ratio = risk_ratio;
    a.nb = l.nb_idx; a.prop = e->prop; a.cap = l.nb_cap; a.entered = e->entered;
    a.result = (int64_t*)ctx->d_scratch;
    a.prev_prop = e->prop_count;
    a.max_pops = (uint64_t)l.w * l.w;
    // crisk is scratch between two risk dilations (dymu_local_expand_risk rebuilds it)
    a.ltot_cache = l.crisk;
    a.axis_d2 = l.axis_d2;
    a.axis_node = l.axis_node;
    {
        size_t cells = (size_t)l.w * l.w;
        uint32_t grid = (uint32_t)std::min<size_t>((cells + 255) / 256, (size_t)ctx->sm_count * 8);
        k_local_total_cost_cache<<<grid, 256, 0, ctx->stream>>>(a.v, l.crisk);
        ctx->launches++;
        DYMU_CUDA_TRY(ctx, cudaGetLastError());
    }
    DYMU_CUDA_TRY(ctx, cudaFuncSetAttribute(k_local_march, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)kBandSmem));
    k_local_march<<<1, 64, kBandSmem, ctx->stream>>>(a);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    int64_t* h = (int64_t*)ctx->h_pinned;
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(h, a.result, 13 * sizeof(int64_t), cudaMemcpyDeviceToHost,
                                       ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (getenv("DYMU_TRACE_CALLS"))
    {
        fprintf(stderr, "[dymu]   march: status %lld, %lld nodes closed, %lld propagated, band peak %lld\n",
                (long long)h[1], (long long)h[2], (long long)h[3], (long long)h[4]);
#ifdef DYMU_LOCAL_PROFILE
        fprintf(stderr, "[dymu]   cycles: end/housekeeping %lld, argmin %lld, neighbours %lld, push %lld\n",
                (long long)h[5], (long long)h[6], (long long)h[7], (long long)h[8]);
        fprintf(stderr, "[dymu]   lane 0 inside neighbours: to loads issued %lld, parent check %lld, state wait %lld, update %lld\n",
                (long long)h[9], (long long)h[10], (long long)h[11], (long long)h[12]);
#endif
    }
    *end_cell = h[0];
    *status = (uint32_t)h[1];
    if (n_closed) *n_closed = (uint64_t)h[2];
    e->prop_count = (uint32_t)h[3];
    if (h[1] == DYMU_LOCAL_WINDOW_EXCEEDED)
    {
        // the march stopped in the middle of a pop: lanes may already have lowered deviations of
        // cells that were never pushed, so the propagated-node list does not cover what was
        // touched.  Put the whole window back to "never propagated"; the caller grows the window
        // and marches again.
        DYMU_TRY(local_reset_wave(ctx));
    }
    return DYMU_OK;
}

int dymu_local_extract_path(dymu_ctx* ctx, int64_t end_cell, double start_x, double start_y,
                            double offset_x, double offset_y, double* out, uint32_t cap,
                            uint32_t* n_out, int* status)
{
    DYMU_GUARD(ctx);
    CallTrace call_trace(__func__);
    if (!ctx || !ctx->loc.allocated || !out || !n_out || !status || cap == 0) return DYMU_ERR_ARG;
    const dymu_local& l = ctx->loc;
    if (end_cell < 0 || end_cell >= (int64_t)l.w * l.w) return DYMU_ERR_ARG;
    size_t out_bytes = (size_t)cap * 6 * sizeof(double);
    DYMU_TRY(dymu_internal_scratch(ctx, 64 + out_bytes, 64));
    LPathArgs a;
    a.v = make_view(ctx);
    a.end_cell = end_cell;
    a.sx = start_x; a.sy = start_y;
    a.off_x = offset_x; a.off_y = offset_y;
    a.out = (double*)((char*)ctx->d_scratch + 64);
    a.cap = cap;
    a.result = (uint32_t*)ctx->d_scratch;
    k_local_path<<<1, 32, 0, ctx->stream>>>(a);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    uint32_t* h = (uint32_t*)ctx->h_pinned;
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(h, a.result, 8, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *n_out = h[0];
    *status = (int)h[1];
    if (h[0])
    {
        DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(out, a.out, (size_t)h[0] * 6 * sizeof(double),
                                           cudaMemcpyDeviceToHost, ctx->stream));
        DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return DYMU_OK;
}

int dymu_local_sample_risk(dymu_ctx* ctx, const double* xy, uint32_t n, double* risk_out)
{
    DYMU_GUARD(ctx);
    CallTrace call_trace(__func__);
    if (!ctx || !ctx->loc.allocated || !xy || !risk_out) return DYMU_ERR_ARG;
    if (n == 0) return DYMU_OK;
    size_t need = (size_t)n * 24;
    DYMU_TRY(dymu_internal_scratch(ctx, need, need));
    memcpy(ctx->h_pinned, xy, (size_t)n * 16);
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_scratch, ctx->h_pinned, (size_t)n * 16,
                                       cudaMemcpyHostToDevice, ctx->stream));
    double* d_out = (double*)((char*)ctx->d_scratch + (size_t)n * 16);
    k_sample_risk<<<dymu_div_up(n, 128), 128, 0, ctx->stream>>>(make_view(ctx),
                                                                (const double*)ctx->d_scratch, n, d_out);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(risk_out, d_out, (size_t)n * 8, cudaMemcpyDeviceToHost,
                                       ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DYMU_OK;
}

int dymu_local_read_entered(dymu_ctx* ctx, uint8_t* host, int clear)
{
    DYMU_GUARD(ctx);
    CallTrace call_trace(__func__);
    if (!ctx || !ctx->loc.allocated || !host) return DYMU_ERR_ARG;
    dymu_local& l = ctx->loc;
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(host, l.entered, (size_t)l.wg * l.wg, cudaMemcpyDeviceToHost,
                                       ctx->stream));
    if (clear) DYMU_CUDA_TRY(ctx, cudaMemsetAsync(l.entered, 0, (size_t)l.wg * l.wg, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DYMU_OK;
}

int dymu_local_cell_of(dymu_ctx* ctx, double x, double y, int64_t* cell)
{
    DYMU_GUARD(ctx);
    CallTrace call_trace(__func__);
    if (!ctx || !ctx->loc.allocated || !cell) return DYMU_ERR_ARG;
    k_cell_of<<<1, 1, 0, ctx->stream>>>(make_view(ctx), x, y, (int64_t*)ctx->d_scratch);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(cell, ctx->d_scratch, 8, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (*cell < 0) *cell = -1;
    return DYMU_OK;
}

}  // extern "C"
