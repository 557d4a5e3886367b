// dymu_path.cu -- gradient-descent waypoint extraction on the device-resident total-cost
// plane (reference: computeGlobalPath / computeNextGlobalWaypoint / gradientNode /
// interpolate, src/DyMu_GlobalPathPlanning.cpp:615-784).
//
// The descent is a sequential chain (each waypoint depends on the previous one), so it is
// latency-bound, not bandwidth-bound: one warp walks one path.  The walker reads a
// PATCH x PATCH window in shared memory that holds the elevation and the normalised node
// gradients of gradientNode, so a step is twelve shared-memory reads and three bilinear
// interpolations; the square root and the two divisions per node are off the per-step chain.
// Only the position is carried from one step to the next: the exit tests of a step (goal,
// grid, window, capacity, and the stall test of the step before) are all decided in one
// branch at the end of the step, whose predicates were ready long before, and a step whose
// cell lies outside the window reads a clamped window cell and is discarded.  Seven helper
// warps build the windows: while the walker walks in one, they build the next one (two
// buffers) where the walker will leave the current one if it keeps its direction.  When the
// stencil leaves the window the walker switches buffers; when the prediction missed (a turn)
// it has the helpers build a window around its cell and waits.  Every lane of the walker
// carries the identical waypoint state (no divergence); lane 0 stores the waypoint.  Batches
// of queries run one CTA per query.
// With slope anisotropy on (dymu_set_anisotropy) the helpers put the characteristic direction
// of the anisotropic metric into the window instead of the normalised gradient; the walker is
// the same.
#include <limits.h>
#include <type_traits>
#include <stdio.h>
#include <stdlib.h>

#include "dymu_ctx.cuh"

namespace
{
constexpr int PATCH = 64;  // cells per window edge
constexpr int P2 = PATCH * PATCH;
constexpr int WIN_DOUBLES = 3 * P2;  // gx, gy, elevation: 96 KB per window, two windows
constexpr size_t PATH_SMEM = 2 * WIN_DOUBLES * sizeof(double);
constexpr int PATCH_LEAD = 20;  // how far a new window is placed ahead of the walker
constexpr int PATH_THREADS = 256;  // warp 0 walks the path; warps 1-7 build windows
constexpr int HELPERS = PATH_THREADS - 32;
constexpr int BUILD_BATCH = 4;  // nodes per helper thread whose loads are in flight together
constexpr int BAR_CMD = 1, BAR_DONE = 2;  // named barriers of the window hand-off

struct PathArgs
{
    const double* T;
    const double* elev;
    uint32_t pitch, nx, ny;
    double gres, tau;
    double x0, y0;
    uint32_t goal_i, goal_j;
    double* out;       // 5 doubles per waypoint
    uint32_t cap;
    uint32_t* result;  // [0] n_out, [1] status
#ifdef DYMU_PATH_PROFILE
    unsigned long long* prof;  // walk cycles, window cycles, windows, missed prefetches (single calls)
#endif
};

// the anisotropic descent also reads the directional-cost planes (order i-1, i+1, j-1, j+1)
struct PathArgsAniso : PathArgs
{
    const double* A;
    size_t a_stride;  // doubles between two of those planes
};

// per-axis rule of gradientNode (G.cpp:722-761); lo/hi missing = NULL neighbour
__device__ __forceinline__ double grad_axis(double f, bool has_lo, double flo, bool has_hi,
                                            double fhi)
{
    const double inf = DYMU_INF;
    if ((!has_lo && !has_hi) || (has_lo && has_hi && flo == inf && fhi == inf)) return 0;
    if (!has_lo || flo == inf)
    {
        if (!has_hi) return 0;  // reference dereferences NULL here
        return fhi - f;
    }
    if (!has_hi || fhi == inf) return f - flo;
    return (fhi - flo) * 0.5;
}

// Window hand-off.  The walker writes the command, then arrives at BAR_CMD, where the helpers
// wait; they build window `buf` at origin (x0, y0) and arrive at BAR_DONE, where the walker
// waits before it reads that window.  Every command but the last is waited for.  x0 = INT_MIN
// tells the helpers to exit; `stop` cuts a build short once the walk has ended.
struct WinCmd
{
    int x0, y0, buf, stop;
};

__device__ __forceinline__ void bar_arrive(int id)
{
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "n"(PATH_THREADS) : "memory");
}
__device__ __forceinline__ void bar_sync(int id)
{
    asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(PATH_THREADS) : "memory");
}

// helper warps: elevation and the normalised gradient of gradientNode (G.cpp:718-772) of
// every node of the window at (x0, y0) whose stencil is inside it; the total cost is read from
// L2.  A thread puts the loads of BUILD_BATCH nodes in flight before it computes any of them.
// ANISO: each difference is scaled by 1/a^2 of the move against it -- a(x->i-1) when it is
// positive, a(x->i+1) otherwise, likewise for y -- before the normalisation; a component that is
// 0 or whose cost is +inf (a neighbour outside the grid) is 0.  (p_x/a_x^2, p_y/a_y^2) is the
// characteristic direction of the metric; with f = 1 it is the normalised gradient up to
// rounding.  An impassable node (all four costs +inf) has no metric and keeps the gradient.
template <bool ANISO, class Args>
__device__ __forceinline__ void build_window(const Args& a, double* wb, int x0, int y0,
                                             const volatile int* stop)
{
    const int t = threadIdx.x - 32;
    for (int k0 = 0; k0 < P2; k0 += BUILD_BATCH * HELPERS)
    {
        if (*stop) return;
        double f[BUILD_BATCH], fl[BUILD_BATCH], fr[BUILD_BATCH], fd[BUILD_BATCH], fu[BUILD_BATCH];
        double ev[BUILD_BATCH];
        double axm[BUILD_BATCH], axp[BUILD_BATCH], aym[BUILD_BATCH], ayp[BUILD_BATCH];
        bool hl[BUILD_BATCH], hr[BUILD_BATCH], hd[BUILD_BATCH], hu[BUILD_BATCH], inner[BUILD_BATCH];
#pragma unroll
        for (int u = 0; u < BUILD_BATCH; ++u)
        {
            const int k = k0 + u * HELPERS + t;
            const int r = k / PATCH, c = k % PATCH;
            const int gx = x0 + c, gy = y0 + r;
            const bool in_grid = k < P2 && gx >= 0 && gy >= 0 && gx < (int)a.nx && gy < (int)a.ny;
            inner[u] = in_grid && r >= 1 && c >= 1 && r < PATCH - 1 && c < PATCH - 1;
            hl[u] = gx > 0;
            hr[u] = gx + 1 < (int)a.nx;
            hd[u] = gy > 0;
            hu[u] = gy + 1 < (int)a.ny;
            const size_t at = in_grid ? (size_t)gy * a.pitch + gx : 0;
            ev[u] = in_grid ? a.elev[at] : 0.0;
            f[u] = fl[u] = fr[u] = fd[u] = fu[u] = 0;
            if (inner[u])
            {
                const double* Tc = a.T + at;
                f[u] = __ldcg(Tc);
                if (hl[u]) fl[u] = __ldcg(Tc - 1);
                if (hr[u]) fr[u] = __ldcg(Tc + 1);
                if (hd[u]) fd[u] = __ldcg(Tc - a.pitch);
                if (hu[u]) fu[u] = __ldcg(Tc + a.pitch);
                if constexpr (ANISO)
                {
                    axm[u] = __ldg(a.A + at);
                    axp[u] = __ldg(a.A + a.a_stride + at);
                    aym[u] = __ldg(a.A + 2 * a.a_stride + at);
                    ayp[u] = __ldg(a.A + 3 * a.a_stride + at);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < BUILD_BATCH; ++u)
        {
            const int k = k0 + u * HELPERS + t;
            double dnx = 0, dny = 0;
            if (inner[u])
            {
                double dx = grad_axis(f[u], hl[u], fl[u], hr[u], fr[u]);
                double dy = grad_axis(f[u], hd[u], fd[u], hu[u], fu[u]);
                if constexpr (ANISO)
                {
                    const double inf = DYMU_INF;
                    if (!(axm[u] == inf && axp[u] == inf && aym[u] == inf && ayp[u] == inf))
                    {
                        const double ax = dx > 0 ? axm[u] : axp[u], ay = dy > 0 ? aym[u] : ayp[u];
                        dx = (dx == 0 || ax == inf) ? 0.0 : dx / (ax * ax);
                        dy = (dy == 0 || ay == inf) ? 0.0 : dy / (ay * ay);
                    }
                }
                if (!((dx == 0) && (dy == 0)))
                {
                    const double nrm = sqrt(dx * dx + dy * dy);
                    dnx = dx / nrm;
                    dny = dy / nrm;
                }
            }
            if (k < P2)
            {
                wb[k] = dnx;
                wb[P2 + k] = dny;
                wb[2 * P2 + k] = ev[u];
            }
        }
    }
}

// origin of a window around cell (cx, cy), PATCH_LEAD cells ahead along (dirx, diry)
__device__ __forceinline__ void place_window(int cx, int cy, double dirx, double diry, int& x0, int& y0)
{
    const double m = fmax(fabs(dirx), fabs(diry));
    int lx = 0, ly = 0;
    if (m > 0)  // false for NaN and for no direction
    {
        lx = (int)(PATCH_LEAD * (dirx / m));
        ly = (int)(PATCH_LEAD * (diry / m));
    }
    x0 = cx - PATCH / 2 + lx;
    y0 = cy - PATCH / 2 + ly;
}

// The next window to build: placed where the walker at grid position (gx, gy) would leave
// the window at (x0, y0) if it kept going along (dirx, diry).
__device__ __forceinline__ void predict_window(double gx, double gy, double dirx, double diry, int x0,
                                               int y0, int& px0, int& py0)
{
    if (!(dirx == dirx) || !(diry == diry)) dirx = diry = 0;
    // the stencil of cell c is inside while x0 + 1 <= c <= x0 + PATCH - 3
    double t = 1e30;
    if (dirx > 0) t = fmin(t, ((double)(x0 + PATCH - 2) - gx) / dirx);
    if (dirx < 0) t = fmin(t, (gx - (double)(x0 + 1)) / -dirx);
    if (diry > 0) t = fmin(t, ((double)(y0 + PATCH - 2) - gy) / diry);
    if (diry < 0) t = fmin(t, (gy - (double)(y0 + 1)) / -diry);
    if (!(t < 1e30)) t = 0;
    t = fmax(t, 0.0);
    place_window((int)floor(gx + t * dirx), (int)floor(gy + t * diry), dirx, diry, px0, py0);
}

// One step of computeNextGlobalWaypoint (G.cpp:666-714) from waypoint (wx, wy) in the window
// at wb / (x0, y0).  The outputs are meaningful when the cell is in the grid and its stencil in
// the window; otherwise the step reads a clamped window cell and the caller discards it.
struct Step
{
    double z, dCx, dCy, nx, ny, gx, gy;
    int cx, cy;
    bool outside, inwin;
};

template <bool UNIT_RES>
__device__ __forceinline__ void walk_step(const PathArgs& a, const double* wb, int x0, int y0, double wx,
                                          double wy, double c_step, double lim_x, double lim_y, Step& s)
{
    // x / 1.0 == x exactly: the usual global_res = 1 gets its own instantiation without the
    // two fp64 divisions (as a run-time select the compiler still evaluated them every step)
    const double gx = UNIT_RES ? wx : wx / a.gres, gy = UNIT_RES ? wy : wy / a.gres;
    s.gx = gx;
    s.gy = gy;
    s.outside = !(gx >= 0.0) || !(gy >= 0.0) || !(gx < lim_x) || !(gy < lim_y);
    // in the grid, trunc(g) is the reference's (double)(uint32_t)g
    const int cx = __double2int_rz(gx), cy = __double2int_rz(gy);
    const double da = gx - trunc(gx), db = gy - trunc(gy);
    s.cx = cx;
    s.cy = cy;
    // stencil [cx-1, cx+2] x [cy-1, cy+2] inside the window <=> 1 <= cx - x0 <= PATCH - 3
    const int lx = (int)((unsigned)cx - (unsigned)x0), ly = (int)((unsigned)cy - (unsigned)y0);
    const int kx = min(max(lx, 1), PATCH - 3), ky = min(max(ly, 1), PATCH - 3);
    s.inwin = (kx == lx) && (ky == ly);
    // corners n00 = (cx, cy), n10 = (cx+1, cy), n01 = (cx, cy+1), n11 = (cx+1, cy+1)
    const double* g = wb + ky * PATCH + kx;
    const double gx00 = g[0], gx10 = g[1], gx01 = g[PATCH], gx11 = g[PATCH + 1];
    const double gy00 = g[P2], gy10 = g[P2 + 1], gy01 = g[P2 + PATCH], gy11 = g[P2 + PATCH + 1];
    const double e00 = g[2 * P2], e10 = g[2 * P2 + 1], e01 = g[2 * P2 + PATCH], e11 = g[2 * P2 + PATCH + 1];
    s.dCx = dymu_interp(da, db, gx00, gx01, gx10, gx11);
    s.dCy = dymu_interp(da, db, gy00, gy01, gy10, gy11);
    // elevation corners are passed as (e00, e10, e01, e11) into (g00, g01, g10, g11):
    // the reference's swapped order, G.cpp:699-704
    s.z = dymu_interp(da, db, e00, e10, e01, e11);
    // a.gres * a.tau * dC in the reference: (gres * tau) is c_step
    s.nx = wx - c_step * s.dCx;
    s.ny = wy - c_step * s.dCy;
}

// The reference compares sqrt(d2) with a constant twice per step (G.cpp:633, 649).  sqrt is
// correctly rounded and monotone, so "sqrt(d2) > c" is "d2 > hi(c)" with hi(c) the largest
// double whose root does not exceed c, and "sqrt(d2) < c" is "d2 < lo(c)" with lo(c) the
// smallest double whose root reaches c.  Both thresholds are found once per path; the
// per-step tests are then exact without a square root on the dependency chain.
__device__ __forceinline__ double dist2(double ax, double ay, double bx, double by)
{
    return (ax - bx) * (ax - bx) + (ay - by) * (ay - by);
}
__device__ __forceinline__ double next_up(double x) { return __longlong_as_double(__double_as_longlong(x) + 1); }
__device__ __forceinline__ double next_down(double x) { return __longlong_as_double(__double_as_longlong(x) - 1); }
__device__ double sqrt_gt_threshold(double c)
{
    if (!(c > 0)) return (c == 0) ? 0.0 : -1.0;  // sqrt(x) > 0 <=> x > 0; any x >= 0 beats a negative c
    double t = c * c;
    while (sqrt(t) > c) t = next_down(t);
    while (sqrt(next_up(t)) <= c) t = next_up(t);
    return t;  // sqrt(x) > c  <=>  x > t
}
__device__ double sqrt_lt_threshold(double c)
{
    if (!(c > 0)) return 0.0;  // sqrt(x) < c never holds
    double t = c * c;
    while (sqrt(t) < c) t = next_up(t);
    while (t > 0 && sqrt(next_down(t)) >= c) t = next_down(t);
    return t;  // sqrt(x) < c  <=>  x < t
}

// computeGlobalPath, G.cpp:615-662
template <bool UNIT_RES, bool ANISO = false, class Args = std::conditional_t<ANISO, PathArgsAniso, PathArgs>>
__global__ void __launch_bounds__(PATH_THREADS, 1) k_global_path(const Args* args_arr)
{
    const Args a = args_arr[blockIdx.x];
    extern __shared__ __align__(16) double path_smem[];  // two windows of WIN_DOUBLES
    __shared__ WinCmd cmd;
    if (threadIdx.x >= 32)
    {
        // helper warps: build windows until the walker signals the end
        for (;;)
        {
            bar_sync(BAR_CMD);
            const int x0 = cmd.x0, y0 = cmd.y0, buf = cmd.buf;
            if (x0 == INT_MIN) return;
            build_window<ANISO>(a, path_smem + buf * WIN_DOUBLES, x0, y0, &cmd.stop);
            bar_arrive(BAR_DONE);
        }
    }
    const int lane = threadIdx.x;
#ifdef DYMU_PATH_PROFILE
    const long long prof_t0 = clock64();
    long long win_cycles = 0;
    unsigned long long windows = 0, misses = 0;
#define PATH_PROF(stmt) stmt
#else
#define PATH_PROF(stmt)
#endif
    auto command = [&](int buf, int x0, int y0) {
        if (lane == 0)
        {
            cmd.x0 = x0;
            cmd.y0 = y0;
            cmd.buf = buf;
        }
        __syncwarp();
        bar_arrive(BAR_CMD);
    };
    if (lane == 0) cmd.stop = 0;

    const double sx = a.gres * (double)a.goal_i, sy = a.gres * (double)a.goal_j;
    const double c_step = a.gres * a.tau;
    const double lim_x = (double)(a.nx - 1), lim_y = (double)(a.ny - 1);
    uint32_t n = 0, status = DYMU_PATH_OK;
    double wx = a.x0, wy = a.y0;
    int cur = 0, x0, y0;  // the window the walker reads: buffer and origin
    int pf_x0, pf_y0;     // the window the helpers build (or built) in buffer cur ^ 1
    bool pending = false;
    Step s;

    auto store = [&](const Step& st, double x, double y) {
        if (lane == 0)
        {
            double* o = a.out + (size_t)5 * n;
            o[0] = x; o[1] = y; o[2] = st.z; o[3] = st.dCx; o[4] = st.dCy;
        }
        n++;
    };

    // first waypoint (G.cpp:620-630): no goal or stall test, a NaN step is its own status
    const double g0x = UNIT_RES ? wx : wx / a.gres, g0y = UNIT_RES ? wy : wy / a.gres;
    if (!(g0x >= 0.0) || !(g0y >= 0.0) || !(g0x < lim_x) || !(g0y < lim_y))
        status = DYMU_PATH_OUTSIDE;
    else
    {
        PATH_PROF(long long t0 = clock64());
        place_window((int)g0x, (int)g0y, 0.0, 0.0, x0, y0);
        command(cur, x0, y0);
        bar_sync(BAR_DONE);
        PATH_PROF(win_cycles += clock64() - t0; windows++; misses++);
        walk_step<UNIT_RES>(a, path_smem, x0, y0, wx, wy, c_step, lim_x, lim_y, s);
        if (isnan(s.nx) || isnan(s.ny)) status = DYMU_PATH_NAN;
        else
        {
            store(s, wx, wy);
            predict_window(s.gx, s.gy, -s.dCx, -s.dCy, x0, y0, pf_x0, pf_y0);
            command(cur ^ 1, pf_x0, pf_y0);
            pending = true;
            const double far2 = sqrt_gt_threshold(2.0 * a.gres);            // dist > 2 * global_res
            const double stall2 = sqrt_lt_threshold(0.01 * a.tau * a.gres);  // dist < 0.01 * tau * global_res
            // previous waypoint (for the stall test, G.cpp:649) and direction of its step; the
            // first waypoint has no stall test: NaN compares false
            double px = NAN, py = NAN, dirx = -s.dCx, diry = -s.dCy;
            wx = s.nx;
            wy = s.ny;
            for (;;)
            {
                walk_step<UNIT_RES>(a, path_smem + cur * WIN_DOUBLES, x0, y0, wx, wy, c_step, lim_x, lim_y, s);
                const bool stalled = dist2(px, py, wx, wy) < stall2;
                // a NaN position ends the reference's while loop (sqrt(NaN) > x is false) and
                // the goal is appended: same here
                const bool at_goal = !(dist2(wx, wy, sx, sy) > far2);
                const bool full = n >= a.cap;
                if (stalled | at_goal | s.outside | !s.inwin | full)
                {
                    // the reference's order: the previous step's stall test ended its loop;
                    // then the loop condition, the grid test, the window, the capacity
                    if (stalled) { status = DYMU_PATH_STALLED; break; }
                    if (at_goal) break;
                    if (s.outside) { status = DYMU_PATH_OUTSIDE; break; }
                    if (!s.inwin)
                    {
                        PATH_PROF(long long t0 = clock64());
                        bar_sync(BAR_DONE);  // the prefetch
                        const bool hit = s.cx - 1 >= pf_x0 && s.cy - 1 >= pf_y0 && s.cx + 2 < pf_x0 + PATCH
                                         && s.cy + 2 < pf_y0 + PATCH;
                        if (!hit)
                        {
                            place_window(s.cx, s.cy, dirx, diry, pf_x0, pf_y0);
                            command(cur ^ 1, pf_x0, pf_y0);
                            bar_sync(BAR_DONE);
                            PATH_PROF(misses++);
                        }
                        cur ^= 1;
                        x0 = pf_x0;
                        y0 = pf_y0;
                        predict_window(s.gx, s.gy, dirx, diry, x0, y0, pf_x0, pf_y0);
                        command(cur ^ 1, pf_x0, pf_y0);
                        PATH_PROF(win_cycles += clock64() - t0; windows++);
                        continue;  // the same step again, in the new window
                    }
                    status = DYMU_PATH_CAPACITY;
                    break;
                }
                store(s, wx, wy);
                px = wx;
                py = wy;
                dirx = -s.dCx;
                diry = -s.dCy;
                wx = s.nx;
                wy = s.ny;
            }
        }
    }
    if (pending)
    {
        if (lane == 0) *(volatile int*)&cmd.stop = 1;
        __syncwarp();
        bar_sync(BAR_DONE);
    }
    command(0, INT_MIN, 0);  // release the helper warps
#ifdef DYMU_PATH_PROFILE
    if (lane == 0 && a.prof)
    {
        a.prof[0] = (unsigned long long)(clock64() - prof_t0 - win_cycles);
        a.prof[1] = (unsigned long long)win_cycles;
        a.prof[2] = windows;
        a.prof[3] = misses;
    }
#endif
    if (lane == 0)
    {
        a.result[0] = n;
        a.result[1] = status;
    }
}

template <class Args> int launch_paths_as(dymu_ctx* ctx, uint32_t n, const Args* d_args)
{
    constexpr bool aniso = std::is_same<Args, PathArgsAniso>::value;
    auto kernel = (ctx->gres == 1.0) ? k_global_path<true, aniso> : k_global_path<false, aniso>;
    DYMU_CUDA_TRY(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PATH_SMEM));
    kernel<<<n, PATH_THREADS, PATH_SMEM, ctx->stream>>>(d_args);
    return DYMU_OK;
}

// d_args: n argument blocks of args_size(ctx) bytes each
int launch_paths(dymu_ctx* ctx, uint32_t n, const void* d_args)
{
    if (ctx->aniso_n) return launch_paths_as(ctx, n, (const PathArgsAniso*)d_args);
    return launch_paths_as(ctx, n, (const PathArgs*)d_args);
}

size_t args_size(const dymu_ctx* ctx) { return ctx->aniso_n ? sizeof(PathArgsAniso) : sizeof(PathArgs); }

// the argument block of one query in the form the kernel of the context's mode takes
void put_args(const dymu_ctx* ctx, const PathArgs& a, void* dst)
{
    if (ctx->aniso_n)
    {
        PathArgsAniso x;
        static_cast<PathArgs&>(x) = a;
        x.A = ctx->dircost;
        x.a_stride = (size_t)ctx->pitch * ctx->rows;
        memcpy(dst, &x, sizeof(x));
    }
    else
        memcpy(dst, &a, sizeof(a));
}
}  // namespace

extern "C" {

int dymu_extract_global_path(dymu_ctx* ctx, uint32_t slot, double x0, double y0, double tau,
                             uint32_t goal_i, uint32_t goal_j, double* out, uint32_t cap,
                             uint32_t* n_out, int* status)
{
    DYMU_GUARD(ctx);
    if (!ctx || !out || !n_out || !status || cap == 0 || slot >= ctx->n_slots) return DYMU_ERR_ARG;
    if (goal_i >= ctx->nx || goal_j >= ctx->ny) return DYMU_ERR_ARG;
    size_t out_bytes = (size_t)cap * 5 * sizeof(double);
    size_t hdr = 256;
    if (ctx->aniso_n) DYMU_TRY(dymu_internal_refresh_ceff(ctx));  // the directional costs are current
    DYMU_TRY(dymu_internal_scratch(ctx, hdr + out_bytes, hdr + out_bytes));
    const size_t asz = args_size(ctx);
    PathArgs a;
    a.T = ctx->T + (size_t)slot * ctx->pitch * ctx->rows;
    a.elev = ctx->elev;
    a.pitch = ctx->pitch; a.nx = ctx->nx; a.ny = ctx->ny;
    a.gres = ctx->gres; a.tau = tau; a.x0 = x0; a.y0 = y0;
    a.goal_i = goal_i; a.goal_j = goal_j;
    a.out = (double*)((char*)ctx->d_scratch + hdr);
    a.cap = cap;
    a.result = (uint32_t*)((char*)ctx->d_scratch + asz);
#ifdef DYMU_PATH_PROFILE
    a.prof = (unsigned long long*)((char*)ctx->d_scratch + asz + 8);
    static_assert(sizeof(PathArgsAniso) + 8 + 4 * 8 <= 256, "path header overflow");
#else
    static_assert(sizeof(PathArgsAniso) + 8 <= 256, "path header overflow");
#endif
    put_args(ctx, a, ctx->h_pinned);
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_scratch, ctx->h_pinned, asz, cudaMemcpyHostToDevice, ctx->stream));
    DYMU_TRY(launch_paths(ctx, 1, ctx->d_scratch));
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    uint32_t* h_res = (uint32_t*)((char*)ctx->h_pinned + asz);
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(h_res, a.result, 8, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *n_out = h_res[0];
    *status = (int)h_res[1];
#ifdef DYMU_PATH_PROFILE
    if (getenv("DYMU_TRACE_CALLS"))
    {
        unsigned long long* h_prof = (unsigned long long*)((char*)ctx->h_pinned + asz + 8);
        DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(h_prof, a.prof, 4 * 8, cudaMemcpyDeviceToHost, ctx->stream));
        DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        fprintf(stderr, "[dymu]   path: %u waypoints, walk %llu cycles, windows %llu cycles for %llu windows "
                "(%llu built while the walker waited)\n", h_res[0], h_prof[0], h_prof[1], h_prof[2], h_prof[3]);
    }
#endif
    if (h_res[0])
    {
        DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(out, a.out, (size_t)h_res[0] * 5 * sizeof(double),
                                           cudaMemcpyDeviceToHost, ctx->stream));
        DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return DYMU_OK;
}

int dymu_extract_global_path_batch(dymu_ctx* ctx, uint32_t n, const uint32_t* slots,
                                   const double* xy0, double tau, const uint32_t* goal_ij,
                                   double* out, uint32_t cap, uint32_t* n_out, int* status)
{
    DYMU_GUARD(ctx);
    if (!ctx || !slots || !xy0 || !goal_ij || !out || !n_out || !status || n == 0 || cap == 0)
        return DYMU_ERR_ARG;
    for (uint32_t q = 0; q < n; ++q)
        if (slots[q] >= ctx->n_slots || goal_ij[2 * q] >= ctx->nx || goal_ij[2 * q + 1] >= ctx->ny)
            return DYMU_ERR_ARG;
    if (ctx->aniso_n) DYMU_TRY(dymu_internal_refresh_ceff(ctx));  // the directional costs are current
    const size_t asz = args_size(ctx);
    const size_t hdr = (((size_t)n * (asz + 8)) + 255) & ~(size_t)255;
    const size_t out_bytes = (size_t)n * cap * 5 * sizeof(double);
    DYMU_TRY(dymu_internal_scratch(ctx, hdr + out_bytes, hdr));
    char* h_args = (char*)ctx->h_pinned;
    char* d_base = (char*)ctx->d_scratch;
    uint32_t* d_res = (uint32_t*)(d_base + (size_t)n * asz);
    for (uint32_t q = 0; q < n; ++q)
    {
        PathArgs a;
        a.T = ctx->T + (size_t)slots[q] * ctx->pitch * ctx->rows;
        a.elev = ctx->elev;
        a.pitch = ctx->pitch; a.nx = ctx->nx; a.ny = ctx->ny;
        a.gres = ctx->gres; a.tau = tau; a.x0 = xy0[2 * q]; a.y0 = xy0[2 * q + 1];
        a.goal_i = goal_ij[2 * q]; a.goal_j = goal_ij[2 * q + 1];
        a.out = (double*)(d_base + hdr) + (size_t)q * cap * 5;
        a.cap = cap;
        a.result = d_res + 2 * q;
#ifdef DYMU_PATH_PROFILE
        a.prof = nullptr;
#endif
        put_args(ctx, a, h_args + (size_t)q * asz);
    }
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(d_base, h_args, (size_t)n * asz, cudaMemcpyHostToDevice, ctx->stream));
    DYMU_TRY(launch_paths(ctx, n, d_base));
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    uint32_t* h_res = (uint32_t*)((char*)ctx->h_pinned + (size_t)n * asz);
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(h_res, d_res, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    for (uint32_t q = 0; q < n; ++q)
    {
        n_out[q] = h_res[2 * q];
        status[q] = (int)h_res[2 * q + 1];
        if (n_out[q])
            DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(out + (size_t)q * cap * 5,
                                               (double*)(d_base + hdr) + (size_t)q * cap * 5,
                                               (size_t)n_out[q] * 5 * sizeof(double), cudaMemcpyDeviceToHost,
                                               ctx->stream));
    }
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DYMU_OK;
}

}  // extern "C"
