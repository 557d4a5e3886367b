// dymu_planes.cu -- context life cycle, plane I/O and the memory-bound stencil kernels
// of the cost-map pipeline (reference: src/DyMu_GlobalPathPlanning.cpp:109-308, 799-855).
//
// Every kernel here streams each plane once: they are bounded by HBM bandwidth
// (algorithmic bytes per cell are listed next to each kernel and in DESIGN.md).
#include <stdlib.h>

#include "dymu_ctx.cuh"

namespace
{
constexpr int kThreads = 256;

inline int stream_grid(const dymu_ctx* ctx, size_t work_items, int per_thread = 1)
{
    size_t blocks = (work_items + (size_t)kThreads * per_thread - 1) / ((size_t)kThreads * per_thread);
    size_t cap = (size_t)ctx->sm_count * 16;  // grid-stride loops: a few waves per SM
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

__global__ void k_fill_f64(double* __restrict__ p, double v, size_t n)
{
    // 8 B written per cell
    size_t stride = (size_t)gridDim.x * blockDim.x;
    size_t n2 = n / 2;
    double2* p2 = reinterpret_cast<double2*>(p);
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n2; k += stride)
        p2[k] = make_double2(v, v);
    if (blockIdx.x == 0 && threadIdx.x == 0 && (n & 1)) p[n - 1] = v;
}

// setCostMap, G.cpp:109-126.  8 B read + (obstacles only) 17 B written per cell.
__global__ void k_set_cost_map(const double* __restrict__ cost, uint8_t* __restrict__ obst,
                               double* __restrict__ traff, double* __restrict__ haz,
                               uint32_t pitch, uint32_t nx, uint32_t ny)
{
    // the padded plane is walked as double2 (pitch is a multiple of 32 doubles, rows 256 B
    // aligned); padding columns/rows are skipped by the bounds test
    const size_t total2 = (size_t)pitch * ny / 2;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const uint32_t pitch2 = pitch / 2;
    const double2* cost2 = reinterpret_cast<const double2*>(cost);
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < total2; k += stride)
    {
        const uint32_t i = (uint32_t)(k % pitch2) * 2;
        if (i >= nx) continue;
        const double2 c = cost2[k];
        const size_t q = 2 * k;
        if (c.x <= 0)
        {
            obst[q] = 1;
            traff[q] = 0.0;
            haz[q] = 1.0;
        }
        if (i + 1 < nx && c.y <= 0)
        {
            obst[q + 1] = 1;
            traff[q + 1] = 0.0;
            haz[q + 1] = 1.0;
        }
    }
}

// computeCostMap pass 1+2 fused per node, G.cpp:157-177: terrain border rule
// (G.cpp:162-165), calculateSlope (G.cpp:186-210), calculateNominalCost (G.cpp:217-293)
// and the obstacle feedback (G.cpp:172-176).  Reads 5 elevations (neighbours hit L1/L2),
// one terrain double; writes slope, raw_cost, terrain, obstacle, locmode (+traff/haz on
// obstacles): ~16 B read + 21 B written per cell.
__global__ void k_slope_nominal(const double* __restrict__ elev,
                                const double* __restrict__ terrain_in, size_t ld_t,
                                const double* __restrict__ lut, const double* __restrict__ slopes,
                                int n_slopes, int n_locs, int n_lut, double Cmax, double gres,
                                double* __restrict__ slope, double* __restrict__ raw,
                                uint32_t* __restrict__ terrain, uint8_t* __restrict__ obst,
                                uint8_t* __restrict__ locmode, double* __restrict__ traff,
                                double* __restrict__ haz, uint32_t pitch, uint32_t nx,
                                uint32_t ny)
{
    size_t total = (size_t)nx * ny;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    const double s_front = slopes[0], s_back = slopes[n_slopes - 1];
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += stride)
    {
        uint32_t j = (uint32_t)(k / nx), i = (uint32_t)(k % nx);
        size_t q = (size_t)j * pitch + i;
        // terrain, G.cpp:162-165
        uint32_t terr;
        if ((i == 0) || (j == 0) || (i == nx - 1) || (j == ny - 1)) terr = 0;
        else if (terrain_in) terr = (uint32_t)terrain_in[(size_t)j * ld_t + i];
        else terr = terrain[q];  // LUT-only rebuild: classes already resident
        terrain[q] = terr;
        // slope, G.cpp:186-210 (nb4List[1]=(i-1,j), [2]=(i+1,j), [0]=(i,j-1), [3]=(i,j+1))
        double e = elev[q], dx, dy;
        if (i == 0) dx = (elev[q + 1] - e) / gres;
        else if (i == nx - 1) dx = (e - elev[q - 1]) / gres;
        else dx = (elev[q + 1] - elev[q - 1]) * 0.5 / gres;
        if (j == 0) dy = (elev[q + pitch] - e) / gres;
        else if (j == ny - 1) dy = (e - elev[q - pitch]) / gres;
        else dy = (elev[q + pitch] - elev[q - pitch]) * 0.5 / gres;
        double sl = atan(sqrt(dx * dx + dy * dy));
        slope[q] = sl;
        // nominal cost, G.cpp:217-293; raw_cost was reset to 0 (G.cpp:160)
        double rawc = 0.0;
        bool ob = false;
        uint8_t lm = locmode[q];
        // a terrain class whose rows lie beyond the table (the reference would read past the end of
        // cost_lutable) is impassable like class 0
        const bool off_table = (unsigned long long)(terr + 1) * (unsigned)n_slopes * (unsigned)n_locs
                               > (unsigned long long)n_lut;
        if (terr == 0 || off_table)
        {
            rawc = Cmax;
            ob = true;
        }
        else if (n_slopes == 1)
        {
            double Cdef = lut[terr * n_locs];
            for (int l = 0; l < n_locs; ++l)
            {
                double Cc = lut[terr * n_locs + l];
                if (Cc < Cdef) Cdef = Cc;
            }
            rawc = fmax(rawc, Cdef);
        }
        else
        {
            double sidx = sl * 180 / 3.14159265358979323846 / (s_back - s_front)
                          * (double)(n_slopes - 1);
            if (sidx > (double)(n_slopes - 1))
            {
                rawc = Cmax;
                ob = true;
            }
            else
            {
                double smin = floor(sidx), smax = ceil(sidx);
                double Cdef = Cmax;
                if (n_locs > 1)
                {
                    for (int l = 1; l < n_locs; ++l)  // starts at 1: G.cpp:268
                    {
                        double C1 = lut[terr * n_slopes * n_locs + l * n_slopes + (int)smin];
                        double C2 = lut[terr * n_slopes * n_locs + l * n_slopes + (int)smax];
                        double Cc = C1 + (C2 - C1) * (sidx - smin);
                        if (Cc < Cdef)
                        {
                            Cdef = Cc;
                            rawc = fmax(rawc, Cdef);
                            lm = (uint8_t)l;
                        }
                    }
                }
                else
                {
                    double C1 = lut[terr * n_slopes + (int)smin];
                    double C2 = lut[terr * n_slopes + (int)smax];
                    Cdef = C1 + (C2 - C1) * (sidx - smin);
                    rawc = fmax(rawc, Cdef);
                    lm = 0;
                }
            }
        }
        raw[q] = rawc;
        locmode[q] = lm;
        if (ob) obst[q] = 1;  // sticky, like the reference's isObstacle
        if (ob || obst[q])
        {
            traff[q] = 0.0;
            haz[q] = 1.0;
        }
    }
}

// smoothCost, G.cpp:297-308: seeded with the node's previous cost.  8 B (cost) + raw
// neighbours (one new 8 B line per cell, rest from cache) read, 8 B written.
__global__ void k_smooth_cost(const double* __restrict__ raw, double* __restrict__ cost,
                              uint32_t pitch, uint32_t nx, uint32_t ny)
{
    size_t total = (size_t)nx * ny;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += stride)
    {
        uint32_t j = (uint32_t)(k / nx), i = (uint32_t)(k % nx);
        size_t q = (size_t)j * pitch + i;
        double Csum = cost[q], n = 5;
        // nb4List order: (i,j-1), (i-1,j), (i+1,j), (i,j+1)
        if (j == 0) n--; else Csum += raw[q - pitch];
        if (i == 0) n--; else Csum += raw[q - 1];
        if (i == nx - 1) n--; else Csum += raw[q + 1];
        if (j == ny - 1) n--; else Csum += raw[q + pitch];
        cost[q] = Csum / n;
    }
}

// C term of G.cpp:527-528 for every node; obstacles (never propagation targets,
// G.cpp:395-397) and padding get +inf.  25 B read + 8 B written per cell.
__global__ void k_ceff(const double* __restrict__ cost, const double* __restrict__ haz,
                       const double* __restrict__ traff, const uint8_t* __restrict__ obst,
                       double* __restrict__ ceff, double gres, uint32_t pitch, uint32_t rows,
                       uint32_t nx, uint32_t ny, double* stats)
{
    size_t total = (size_t)pitch * rows;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    double sum = 0, cnt = 0;  // of the finite values: sets the width of the solver's priority band
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += stride)
    {
        uint32_t j = (uint32_t)(q / pitch), i = (uint32_t)(q % pitch);
        double c = DYMU_INF;
        if (i < nx && j < ny && !obst[q])
        {
            c = gres * (cost[q]) * (2 + haz[q] - traff[q]);
            if (c < DYMU_INF)
            {
                sum += c;
                cnt += 1.0;
            }
        }
        ceff[q] = c;
    }
    if (stats)
    {
        for (int o = 16; o > 0; o >>= 1)
        {
            sum += __shfl_down_sync(0xffffffffu, sum, o);
            cnt += __shfl_down_sync(0xffffffffu, cnt, o);
        }
        if ((threadIdx.x & 31) == 0 && cnt > 0)
        {
            atomicAdd(&stats[0], sum);
            atomicAdd(&stats[1], cnt);
        }
    }
}

// sum and count of the finite C_eff values (sets the width of the solver's priority band)
__global__ void k_ceff_stats(const double* __restrict__ ceff, size_t n, double* out)
{
    size_t stride = (size_t)gridDim.x * blockDim.x;
    double sum = 0, cnt = 0;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += stride)
    {
        double c = ceff[q];
        if (c < DYMU_INF)
        {
            sum += c;
            cnt += 1.0;
        }
    }
    for (int o = 16; o > 0; o >>= 1)
    {
        sum += __shfl_down_sync(0xffffffffu, sum, o);
        cnt += __shfl_down_sync(0xffffffffu, cnt, o);
    }
    if ((threadIdx.x & 31) == 0 && cnt > 0)
    {
        atomicAdd(&out[0], sum);
        atomicAdd(&out[1], cnt);
    }
}

// the factor table of the anisotropic solve, passed by value (it lives in the constant bank)
struct AnisoTable
{
    int n;
    double theta[DYMU_ANISO_MAX], f[DYMU_ANISO_MAX];
};

// f(theta): piecewise linear in the table, clamped at both ends (restated by
// the test oracle in the same expression order)
__device__ __forceinline__ double aniso_factor(const AnisoTable& t, double th)
{
    if (th <= t.theta[0]) return t.f[0];
    if (th >= t.theta[t.n - 1]) return t.f[t.n - 1];
    int k = 0;
    while (th >= t.theta[k + 1]) ++k;
    return t.f[k] + (t.f[k + 1] - t.f[k]) * ((th - t.theta[k]) / (t.theta[k + 1] - t.theta[k]));
}

// Directional costs of the anisotropic solve, all four planes of every padded cell:
//     a(x->m) = C_eff(x) * f(atan((elev[m] - elev[x]) / gres) * (180/pi))
// toward m = i-1, i+1, j-1, j+1; +inf where C_eff(x) is +inf (obstacles, padding) and toward a
// neighbour outside the grid.  16 B read + 32 B written per cell (the neighbours' elevations come
// from cache).  Accumulates sum and count of the finite values: the band width of the solver.
__global__ void k_dircost(const double* __restrict__ elev, const double* __restrict__ ceff,
                          double* __restrict__ A, size_t plane, double gres, uint32_t pitch, uint32_t rows,
                          uint32_t nx, uint32_t ny, AnisoTable tab, double* stats)
{
    constexpr double kDeg = 180.0 / 3.141592653589793;
    const size_t total = (size_t)pitch * rows;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    double sum = 0, cnt = 0;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += stride)
    {
        const uint32_t j = (uint32_t)(q / pitch), i = (uint32_t)(q % pitch);
        const double c = ceff[q];
        double a[4] = {DYMU_INF, DYMU_INF, DYMU_INF, DYMU_INF};
        if (c < DYMU_INF && i < nx && j < ny)
        {
            const double e = elev[q];
            const bool has[4] = {i > 0, i + 1 < nx, j > 0, j + 1 < ny};
            const ptrdiff_t off[4] = {-1, 1, -(ptrdiff_t)pitch, (ptrdiff_t)pitch};
#pragma unroll
            for (int d = 0; d < 4; ++d)
                if (has[d])
                {
                    a[d] = c * aniso_factor(tab, atan((elev[q + off[d]] - e) / gres) * kDeg);
                    if (a[d] < DYMU_INF)
                    {
                        sum += a[d];
                        cnt += 1.0;
                    }
                }
        }
#pragma unroll
        for (int d = 0; d < 4; ++d) A[d * plane + q] = a[d];
    }
    for (int o = 16; o > 0; o >>= 1)
    {
        sum += __shfl_down_sync(0xffffffffu, sum, o);
        cnt += __shfl_down_sync(0xffffffffu, cnt, o);
    }
    if ((threadIdx.x & 31) == 0 && cnt > 0)
    {
        atomicAdd(&stats[0], sum);
        atomicAdd(&stats[1], cnt);
    }
}

// Factor planes of the anisotropic map batch (dymu_set_maps_anisotropy): k_dircost's factor alone,
//     F_d(x) = f(atan((elev[m] - elev[x]) / gres) * (180/pi))
// for every cell of the grid toward its neighbour m = i-1, i+1, j-1, j+1, +inf toward a neighbour
// outside the grid and on the padding (never 0: the solver multiplies, and inf * 0 is NaN).  The
// solver's C_q(x) * F_d(x) is then k_dircost's a(x->m) of map q bit for bit.  8 B read + 32 B
// written per cell.
__global__ void k_dirfactor(const double* __restrict__ elev, double* __restrict__ F, size_t plane, double gres,
                            uint32_t pitch, uint32_t rows, uint32_t nx, uint32_t ny, AnisoTable tab)
{
    constexpr double kDeg = 180.0 / 3.141592653589793;
    const size_t total = (size_t)pitch * rows;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += stride)
    {
        const uint32_t j = (uint32_t)(q / pitch), i = (uint32_t)(q % pitch);
        double a[4] = {DYMU_INF, DYMU_INF, DYMU_INF, DYMU_INF};
        if (i < nx && j < ny)
        {
            const double e = elev[q];
            const bool has[4] = {i > 0, i + 1 < nx, j > 0, j + 1 < ny};
            const ptrdiff_t off[4] = {-1, 1, -(ptrdiff_t)pitch, (ptrdiff_t)pitch};
#pragma unroll
            for (int d = 0; d < 4; ++d)
                if (has[d]) a[d] = aniso_factor(tab, atan((elev[q + off[d]] - e) / gres) * kDeg);
        }
#pragma unroll
        for (int d = 0; d < 4; ++d) F[d * plane + q] = a[d];
    }
}

// dense read-back with the getter transforms of G.cpp:799-829.  8(+17) B read, 8 B written.
__global__ void k_readback(const double* __restrict__ src, const double* __restrict__ haz,
                           const double* __restrict__ traff, const uint8_t* __restrict__ obst,
                           double* __restrict__ dst, int xform, uint32_t pitch, uint32_t nx,
                           uint32_t ny)
{
    size_t total = (size_t)nx * ny;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += stride)
    {
        uint32_t j = (uint32_t)(k / nx), i = (uint32_t)(k % nx);
        size_t q = (size_t)j * pitch + i;
        double v = src[q];
        if (xform == DYMU_XFORM_INF_TO_MINUS1)
        {
            if (v == DYMU_INF) v = -1.0;
        }
        else if (xform == DYMU_XFORM_EFFECTIVE_COST)
        {
            if (obst[q]) v = -1.0;
            else v = v * (2 + haz[q] - traff[q]);
        }
        dst[k] = v;
    }
}

__global__ void k_gather_cells(const double* __restrict__ src, uint32_t pitch, uint32_t nx,
                               const uint32_t* __restrict__ idx, uint32_t n,
                               double* __restrict__ out)
{
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n)
    {
        uint32_t j = idx[k] / nx, i = idx[k] % nx;
        out[k] = src[(size_t)j * pitch + i];
    }
}

__global__ void k_read_node(const double* elev, const double* slope, const double* raw,
                            const double* cost, const double* haz, const double* traff,
                            const double* T, const uint32_t* terrain, const uint8_t* obst,
                            const uint8_t* locmode, size_t q, double* out)
{
    out[0] = elev[q]; out[1] = slope[q]; out[2] = raw[q]; out[3] = cost[q]; out[4] = haz[q];
    out[5] = traff[q]; out[6] = T[q]; out[7] = (double)terrain[q]; out[8] = (double)obst[q];
    out[9] = (double)locmode[q];
}

// counts cells with T <= threshold (threshold = +inf counts the finite ones)
__global__ void k_count_finite(const double* __restrict__ T, uint32_t pitch, uint32_t nx,
                               uint32_t ny, double threshold, unsigned long long* out)
{
    size_t total = (size_t)nx * ny;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    unsigned long long c = 0;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += stride)
    {
        uint32_t j = (uint32_t)(k / nx), i = (uint32_t)(k % nx);
        double v = T[(size_t)j * pitch + i];
        c += (v < DYMU_INF && v <= threshold) ? 1 : 0;
    }
    for (int o = 16; o > 0; o >>= 1) c += __shfl_down_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

double* plane_ptr(dymu_ctx* ctx, int plane)
{
    switch (plane)
    {
        case DYMU_PLANE_ELEVATION: return ctx->elev;
        case DYMU_PLANE_SLOPE: return ctx->slope;
        case DYMU_PLANE_RAW_COST: return ctx->raw;
        case DYMU_PLANE_COST: return ctx->cost;
        case DYMU_PLANE_HAZARD_DENSITY: return ctx->haz;
        case DYMU_PLANE_TRAFFICABILITY: return ctx->traff;
        case DYMU_PLANE_TOTAL_COST: return ctx->T;
        case DYMU_PLANE_CEFF: return ctx->ceff;
        case DYMU_PLANE_DIRCOST_XM:
        case DYMU_PLANE_DIRCOST_XP:
        case DYMU_PLANE_DIRCOST_YM:
        case DYMU_PLANE_DIRCOST_YP:
            // only while anisotropy is on
            return ctx->dircost ? ctx->dircost + (size_t)(plane - DYMU_PLANE_DIRCOST_XM) * ctx->pitch * ctx->rows
                                : nullptr;
        case DYMU_PLANE_CLEARANCE: return ctx->clear;  // only while obstacle clearance is on
        default: return nullptr;
    }
}
uint8_t* plane_ptr_u8(dymu_ctx* ctx, int plane)
{
    switch (plane)
    {
        case DYMU_PLANE_U8_OBSTACLE: return ctx->obst;
        case DYMU_PLANE_U8_LOCMODE: return ctx->locmode;
        default: return nullptr;
    }
}

int fill_plane(dymu_ctx* ctx, double* p, double v, size_t n)
{
    k_fill_f64<<<stream_grid(ctx, n / 2 + 1), kThreads, 0, ctx->stream>>>(p, v, n);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    return DYMU_OK;
}

bool is_dircost(int plane) { return plane >= DYMU_PLANE_DIRCOST_XM && plane <= DYMU_PLANE_DIRCOST_YP; }
// planes derived from the others on the device, never written from outside
bool is_read_only(int plane) { return is_dircost(plane) || plane == DYMU_PLANE_CLEARANCE; }

// brings a derived plane up to date before it is read
int refresh_for_read(dymu_ctx* ctx, int plane)
{
    if (plane == DYMU_PLANE_CEFF || is_dircost(plane)) return dymu_internal_refresh_ceff(ctx);
    // the clearance plane alone: C_eff stays dirty for dymu_solve_incremental to compare against
    if (plane == DYMU_PLANE_CLEARANCE) return dymu_internal_clearance_update(ctx);
    return DYMU_OK;
}

// planes C_eff (and, while anisotropy is on, the directional costs) are built from
bool feeds_ceff(const dymu_ctx* ctx, int plane)
{
    return plane == DYMU_PLANE_COST || plane == DYMU_PLANE_HAZARD_DENSITY || plane == DYMU_PLANE_TRAFFICABILITY
           || (ctx->aniso_n && plane == DYMU_PLANE_ELEVATION);
}
}  // namespace

int dymu_internal_fill(dymu_ctx* ctx, double* p, double v, size_t n) { return fill_plane(ctx, p, v, n); }

int dymu_internal_scratch(dymu_ctx* ctx, size_t dev_bytes, size_t host_bytes)
{
    if (dev_bytes > ctx->d_scratch_bytes)
    {
        if (ctx->d_scratch) cudaFree(ctx->d_scratch);
        ctx->d_scratch = nullptr;
        ctx->d_scratch_bytes = 0;
        DYMU_CUDA_TRY(ctx, cudaMalloc(&ctx->d_scratch, dev_bytes));
        ctx->d_scratch_bytes = dev_bytes;
    }
    if (host_bytes > ctx->h_pinned_bytes)
    {
        if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
        ctx->h_pinned = nullptr;
        ctx->h_pinned_bytes = 0;
        DYMU_CUDA_TRY(ctx, cudaMallocHost(&ctx->h_pinned, host_bytes));
        ctx->h_pinned_bytes = host_bytes;
    }
    return DYMU_OK;
}

static int build_dircost(dymu_ctx* ctx);

extern "C" {

int dymu_create(int device, uint32_t nx, uint32_t ny, double global_res, double local_res,
                dymu_ctx** out)
{
    if (!out || nx < 2 || ny < 2 || !(global_res > 0) || !(local_res > 0)) return DYMU_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return DYMU_ERR_NODEVICE;
    dymu_ctx* ctx = (dymu_ctx*)calloc(1, sizeof(dymu_ctx));
    if (!ctx) return DYMU_ERR_ARG;
    if (device < 0) cudaGetDevice(&device);
    ctx->device = device;
    if (device >= ndev)
    {
        free(ctx);
        return DYMU_ERR_NODEVICE;
    }
    dymu_device_guard guard__(device);  // the caller's current device is restored on return
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess)
    {
        free(ctx);
        return DYMU_ERR_NODEVICE;
    }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->nx = nx;
    ctx->ny = ny;
    ctx->gres = global_res;
    ctx->lres = local_res;
    ctx->ntx = dymu_div_up(nx, kTile);
    ctx->nty = dymu_div_up(ny, kTile);
    ctx->pitch = ctx->ntx * kTile;
    ctx->rows = ctx->nty * kTile;
    ctx->n_slots = 1;
    *out = ctx;  // from here on the caller owns ctx and can read the error text
    DYMU_CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    DYMU_CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    DYMU_CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_copy, cudaEventDisableTiming));
    DYMU_CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_part, cudaEventDisableTiming));
    DYMU_CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_part0, cudaEventDisableTiming));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->d_upflag, 4 * sizeof(uint32_t)));
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_upflag, 0, 4 * sizeof(uint32_t), ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaHostAlloc((void**)&ctx->h_upvals, 4 * sizeof(uint32_t), cudaHostAllocDefault));
    for (uint32_t k = 0; k < 4; ++k) ctx->h_upvals[k] = k;
    DYMU_CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_up, cudaEventDisableTiming));
    DYMU_CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_tail, cudaEventDisableTiming));
    DYMU_CUDA_TRY(ctx, cudaEventCreate(&ctx->ev0));
    DYMU_CUDA_TRY(ctx, cudaEventCreate(&ctx->ev1));
    DYMU_CUDA_TRY(ctx, cudaEventCreate(&ctx->ev2));
    size_t n = (size_t)ctx->pitch * ctx->rows;
    double** f64[] = {&ctx->elev, &ctx->slope, &ctx->raw, &ctx->cost, &ctx->haz, &ctx->traff,
                      &ctx->ceff, &ctx->T};
    for (double** p : f64) DYMU_CUDA_TRY(ctx, cudaMalloc((void**)p, n * sizeof(double)));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->terrain, n * sizeof(uint32_t)));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->obst, n));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->locmode, n));
    // globalNode constructor defaults, H.hpp:88-107
    for (double* p : {ctx->elev, ctx->slope, ctx->raw, ctx->cost, ctx->haz})
        DYMU_CUDA_TRY(ctx, cudaMemsetAsync(p, 0, n * sizeof(double), ctx->stream));
    DYMU_TRY(fill_plane(ctx, ctx->traff, 1.0, n));
    DYMU_TRY(fill_plane(ctx, ctx->T, 1.0 / 0.0, n));
    DYMU_TRY(fill_plane(ctx, ctx->ceff, 1.0 / 0.0, n));
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(ctx->terrain, 0, n * sizeof(uint32_t), ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(ctx->obst, 0, n, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(ctx->locmode, 0xFF, n, ctx->stream));
    DYMU_TRY(dymu_internal_scratch(ctx, 1 << 20, 1 << 20));
    DYMU_TRY(dymu_internal_fim_alloc(ctx, &ctx->work, (size_t)ctx->ntx * ctx->nty));
    DYMU_TRY(dymu_internal_fim_configure(ctx));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->ceff_dirty = true;
    return DYMU_OK;
}

int dymu_destroy(dymu_ctx* ctx)
{
    if (!ctx) return DYMU_OK;
    DYMU_GUARD(ctx);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    dymu_internal_local_free(ctx);
    dymu_internal_incremental_free(ctx);
    dymu_internal_clearance_free(ctx);
    dymu_internal_maps_free(ctx);
    dymu_internal_fim_free(&ctx->work);
    void* ptrs[] = {ctx->elev, ctx->slope, ctx->raw, ctx->cost, ctx->haz, ctx->traff, ctx->ceff,
                    ctx->T, ctx->terrain, ctx->obst, ctx->locmode, ctx->d_lut, ctx->d_slopes,
                    ctx->d_stage, ctx->d_scratch, ctx->tile_tmax, ctx->d_upflag, ctx->dircost};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->ev2) cudaEventDestroy(ctx->ev2);
    for (int k = 0; k < 8; ++k)
        if (ctx->user_ev[k]) cudaEventDestroy(ctx->user_ev[k]);
    if (ctx->ev_copy) cudaEventDestroy(ctx->ev_copy);
    if (ctx->ev_part) cudaEventDestroy(ctx->ev_part);
    if (ctx->ev_part0) cudaEventDestroy(ctx->ev_part0);
    if (ctx->h_upvals) cudaFreeHost(ctx->h_upvals);
    if (ctx->ev_up) cudaEventDestroy(ctx->ev_up);
    if (ctx->ev_tail) cudaEventDestroy(ctx->ev_tail);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    dymu_internal_unmark_all(ctx);
    free(ctx);
    return DYMU_OK;
}

const char* dymu_last_error(const dymu_ctx* ctx) { return ctx ? ctx->err : "null context"; }
void* dymu_stream(dymu_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
uint64_t dymu_launch_count(const dymu_ctx* ctx) { return ctx ? ctx->launches : 0; }

int dymu_synchronize(dymu_ctx* ctx)
{
    DYMU_GUARD(ctx);
    if (!ctx) return DYMU_ERR_ARG;
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    // ... and the rest of a direct matrix delivery, which runs on the copy stream
    if (ctx->export_tail_pending) DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy_stream));
    return DYMU_OK;
}

int dymu_event_record(dymu_ctx* ctx, int which)
{
    DYMU_GUARD(ctx);
    if (!ctx || which < 0 || which >= 8) return DYMU_ERR_ARG;
    if (!ctx->user_ev[which]) DYMU_CUDA_TRY(ctx, cudaEventCreate(&ctx->user_ev[which]));
    DYMU_CUDA_TRY(ctx, cudaEventRecord(ctx->user_ev[which], ctx->stream));
    return DYMU_OK;
}

int dymu_event_elapsed_ms(dymu_ctx* ctx, int a, int b, float* ms)
{
    DYMU_GUARD(ctx);
    if (!ctx || !ms || a < 0 || a >= 8 || b < 0 || b >= 8 || !ctx->user_ev[a] || !ctx->user_ev[b])
        return DYMU_ERR_ARG;
    DYMU_CUDA_TRY(ctx, cudaEventSynchronize(ctx->user_ev[b]));
    DYMU_CUDA_TRY(ctx, cudaEventElapsedTime(ms, ctx->user_ev[a], ctx->user_ev[b]));
    return DYMU_OK;
}

int dymu_geometry(const dymu_ctx* ctx, uint32_t* tile, uint32_t* pitch, uint32_t* rows)
{
    if (!ctx) return DYMU_ERR_ARG;
    if (tile) *tile = kTile;
    if (pitch) *pitch = ctx->pitch;
    if (rows) *rows = ctx->rows;
    return DYMU_OK;
}

int dymu_upload_plane(dymu_ctx* ctx, int plane, const double* host, size_t ld)
{
    DYMU_GUARD(ctx);
    if (!ctx || !host || ld < ctx->nx) return DYMU_ERR_ARG;
    if (is_dircost(plane)) DYMU_FAIL(ctx, DYMU_ERR_ARG, "the directional-cost planes are read-only");
    if (plane == DYMU_PLANE_CLEARANCE) DYMU_FAIL(ctx, DYMU_ERR_ARG, "the clearance plane is read-only");
    double* d = plane_ptr(ctx, plane);
    if (!d) DYMU_FAIL(ctx, DYMU_ERR_ARG, "unknown plane %d", plane);
    if (plane == DYMU_PLANE_TOTAL_COST) DYMU_TRY(dymu_internal_settle_delivery(ctx));
    DYMU_CUDA_TRY(ctx, cudaMemcpy2DAsync(d, ctx->pitch * sizeof(double), host, ld * sizeof(double),
                                         ctx->nx * sizeof(double), ctx->ny, cudaMemcpyHostToDevice,
                                         ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (feeds_ceff(ctx, plane)) ctx->ceff_dirty = true;
    if (plane == DYMU_PLANE_TOTAL_COST) ctx->solved = ctx->export_done = false;
    return DYMU_OK;
}

static int ensure_stage(dymu_ctx* ctx)
{
    size_t need = (size_t)ctx->nx * ctx->ny;
    if (ctx->stage_elems < need)
    {
        if (ctx->d_stage) cudaFree(ctx->d_stage);
        ctx->d_stage = nullptr;
        ctx->stage_elems = 0;
        DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->d_stage, need * sizeof(double)));
        ctx->stage_elems = need;
    }
    return DYMU_OK;
}

static int download_f64_on(dymu_ctx* ctx, cudaStream_t st, const double* d, double* host, size_t ld,
                           int xform)
{
    if (xform == DYMU_XFORM_NONE)
    {
        DYMU_CUDA_TRY(ctx, cudaMemcpy2DAsync(host, ld * sizeof(double), d,
                                             ctx->pitch * sizeof(double), ctx->nx * sizeof(double),
                                             ctx->ny, cudaMemcpyDeviceToHost, st));
    }
    else
    {
        DYMU_TRY(ensure_stage(ctx));
        ctx->terrain_staged = false;  // the staging plane is about to be overwritten
        size_t n = (size_t)ctx->nx * ctx->ny;
        k_readback<<<stream_grid(ctx, n), kThreads, 0, st>>>(
            d, ctx->haz, ctx->traff, ctx->obst, ctx->d_stage, xform, ctx->pitch, ctx->nx, ctx->ny);
        ctx->launches++;
        DYMU_CUDA_TRY(ctx, cudaGetLastError());
        DYMU_CUDA_TRY(ctx, cudaMemcpy2DAsync(host, ld * sizeof(double), ctx->d_stage,
                                             ctx->nx * sizeof(double), ctx->nx * sizeof(double),
                                             ctx->ny, cudaMemcpyDeviceToHost, st));
    }
    return DYMU_OK;
}

static int download_f64(dymu_ctx* ctx, const double* d, double* host, size_t ld, int xform)
{
    DYMU_TRY(download_f64_on(ctx, ctx->stream, d, host, ld, xform));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DYMU_OK;
}

int dymu_download_plane(dymu_ctx* ctx, int plane, double* host, size_t ld, int xform)
{
    DYMU_GUARD(ctx);
    if (!ctx || !host || ld < ctx->nx) return DYMU_ERR_ARG;
    DYMU_TRY(refresh_for_read(ctx, plane));
    double* d = plane_ptr(ctx, plane);
    if (!d) DYMU_FAIL(ctx, DYMU_ERR_ARG, "unknown plane %d", plane);
    return download_f64(ctx, d, host, ld, xform);
}

// the solve itself stored the matrix there (dymu_set_total_cost_export)
static bool already_delivered(const dymu_ctx* ctx, uint32_t slot, const double* host, size_t ld, int xform)
{
    return ctx->export_done && slot == 0 && host == ctx->export_host && ld == ctx->export_ld
           && xform == ctx->export_xform;
}

int dymu_set_total_cost_export(dymu_ctx* ctx, double* host, size_t ld, int xform, int* direct)
{
    DYMU_GUARD(ctx);
    if (!ctx) return DYMU_ERR_ARG;
    if (direct) *direct = 0;
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy_stream));  // a delivery that is still running
    ctx->export_tail_pending = false;
    ctx->export_host = ctx->export_dev = nullptr;
    ctx->export_done = false;
    if (!host) return DYMU_OK;
    if (ld < ctx->nx || (xform != DYMU_XFORM_NONE && xform != DYMU_XFORM_INF_TO_MINUS1)) return DYMU_ERR_ARG;
    // page-locked and mapped?  Both ends of the matrix are asked: a buffer that is only partly
    // registered is no use
    cudaPointerAttributes lo, hi;
    const double* last = host + (size_t)(ctx->ny - 1) * ld + (ctx->nx - 1);
    if (cudaPointerGetAttributes(&lo, host) != cudaSuccess || cudaPointerGetAttributes(&hi, last) != cudaSuccess)
    {
        cudaGetLastError();
        return DYMU_OK;
    }
    if (lo.type != cudaMemoryTypeHost || hi.type != cudaMemoryTypeHost || !lo.devicePointer || !hi.devicePointer
        || (const char*)hi.devicePointer - (const char*)lo.devicePointer != (const char*)last - (const char*)host)
        return DYMU_OK;
    ctx->export_host = host;
    ctx->export_dev = (double*)lo.devicePointer;
    ctx->export_ld = ld;
    ctx->export_xform = xform;
    if (direct) *direct = 1;
    return DYMU_OK;
}

int dymu_download_total_cost(dymu_ctx* ctx, uint32_t slot, double* host, size_t ld, int xform)
{
    DYMU_GUARD(ctx);
    if (!ctx || !host || ld < ctx->nx || slot >= ctx->n_slots) return DYMU_ERR_ARG;
    if (already_delivered(ctx, slot, host, ld, xform))
    {
        DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy_stream));  // k_deliver_rest
        return DYMU_OK;
    }
    return download_f64(ctx, ctx->T + (size_t)slot * ctx->pitch * ctx->rows, host, ld, xform);
}

int dymu_download_total_cost_begin(dymu_ctx* ctx, uint32_t slot, double* host, size_t ld, int xform)
{
    DYMU_GUARD(ctx);
    if (!ctx || !host || ld < ctx->nx || slot >= ctx->n_slots) return DYMU_ERR_ARG;
    if (already_delivered(ctx, slot, host, ld, xform)) return DYMU_OK;
    if (xform != DYMU_XFORM_NONE) DYMU_TRY(ensure_stage(ctx));  // allocate before forking
    DYMU_CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_copy, 0));
    return download_f64_on(ctx, ctx->copy_stream, ctx->T + (size_t)slot * ctx->pitch * ctx->rows, host, ld,
                           xform);
}

int dymu_download_total_cost_end(dymu_ctx* ctx)
{
    DYMU_GUARD(ctx);
    if (!ctx) return DYMU_ERR_ARG;
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy_stream));
    // later work on the main stream may overwrite the plane or the staging buffer
    DYMU_CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy, ctx->copy_stream));
    DYMU_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_copy, 0));
    return DYMU_OK;
}

int dymu_download_plane_u8(dymu_ctx* ctx, int plane, uint8_t* host, size_t ld)
{
    DYMU_GUARD(ctx);
    if (!ctx || !host || ld < ctx->nx) return DYMU_ERR_ARG;
    uint8_t* d = plane_ptr_u8(ctx, plane);
    if (!d) DYMU_FAIL(ctx, DYMU_ERR_ARG, "unknown u8 plane %d", plane);
    DYMU_CUDA_TRY(ctx, cudaMemcpy2DAsync(host, ld, d, ctx->pitch, ctx->nx, ctx->ny,
                                         cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DYMU_OK;
}

static bool rect_ok(const dymu_ctx* ctx, uint32_t i0, uint32_t j0, uint32_t w, uint32_t h)
{
    return w > 0 && h > 0 && (uint64_t)i0 + w <= ctx->nx && (uint64_t)j0 + h <= ctx->ny;
}

int dymu_read_rect(dymu_ctx* ctx, int plane, uint32_t i0, uint32_t j0, uint32_t w, uint32_t h,
                   double* host)
{
    DYMU_GUARD(ctx);
    if (!ctx || !host || !rect_ok(ctx, i0, j0, w, h)) return DYMU_ERR_ARG;
    DYMU_TRY(refresh_for_read(ctx, plane));
    double* d = plane_ptr(ctx, plane);
    if (!d) return DYMU_ERR_ARG;
    DYMU_CUDA_TRY(ctx, cudaMemcpy2DAsync(host, w * sizeof(double), d + (size_t)j0 * ctx->pitch + i0,
                                         ctx->pitch * sizeof(double), w * sizeof(double), h,
                                         cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DYMU_OK;
}

int dymu_write_rect(dymu_ctx* ctx, int plane, uint32_t i0, uint32_t j0, uint32_t w, uint32_t h,
                    const double* host)
{
    DYMU_GUARD(ctx);
    if (!ctx || !host || !rect_ok(ctx, i0, j0, w, h) || is_read_only(plane)) return DYMU_ERR_ARG;
    double* d = plane_ptr(ctx, plane);
    if (!d) return DYMU_ERR_ARG;
    if (plane == DYMU_PLANE_TOTAL_COST) DYMU_TRY(dymu_internal_settle_delivery(ctx));
    DYMU_CUDA_TRY(ctx, cudaMemcpy2DAsync(d + (size_t)j0 * ctx->pitch + i0,
                                         ctx->pitch * sizeof(double), host, w * sizeof(double),
                                         w * sizeof(double), h, cudaMemcpyHostToDevice,
                                         ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (feeds_ceff(ctx, plane)) ctx->ceff_dirty = true;
    if (plane == DYMU_PLANE_TOTAL_COST) ctx->solved = ctx->export_done = false;  // no longer the solver's fixed point
    return DYMU_OK;
}

int dymu_read_rect_u8(dymu_ctx* ctx, int plane, uint32_t i0, uint32_t j0, uint32_t w, uint32_t h,
                      uint8_t* host)
{
    DYMU_GUARD(ctx);
    if (!ctx || !host || !rect_ok(ctx, i0, j0, w, h)) return DYMU_ERR_ARG;
    uint8_t* d = plane_ptr_u8(ctx, plane);
    if (!d) return DYMU_ERR_ARG;
    DYMU_CUDA_TRY(ctx, cudaMemcpy2DAsync(host, w, d + (size_t)j0 * ctx->pitch + i0, ctx->pitch, w,
                                         h, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DYMU_OK;
}

int dymu_plane_device_ptr(dymu_ctx* ctx, int plane, void** dptr, size_t* pitch_elems)
{
    DYMU_GUARD(ctx);
    if (!ctx || !dptr || is_read_only(plane)) return DYMU_ERR_ARG;
    double* d = plane_ptr(ctx, plane);
    if (!d) return DYMU_ERR_ARG;
    *dptr = d;
    if (pitch_elems) *pitch_elems = ctx->pitch;
    if (feeds_ceff(ctx, plane)) ctx->ceff_dirty = true;  // the caller may write through the pointer
    return DYMU_OK;
}

int dymu_set_cost_map(dymu_ctx* ctx, const double* host, size_t ld)
{
    DYMU_GUARD(ctx);
    if (!ctx) return DYMU_ERR_ARG;
    if (host)
    {
        if (ld < ctx->nx) return DYMU_ERR_ARG;
        DYMU_CUDA_TRY(ctx, cudaMemcpy2DAsync(ctx->cost, ctx->pitch * sizeof(double), host,
                                             ld * sizeof(double), ctx->nx * sizeof(double), ctx->ny,
                                             cudaMemcpyHostToDevice, ctx->stream));
    }
    size_t n = (size_t)ctx->nx * ctx->ny;
    k_set_cost_map<<<stream_grid(ctx, n), kThreads, 0, ctx->stream>>>(
        ctx->cost, ctx->obst, ctx->traff, ctx->haz, ctx->pitch, ctx->nx, ctx->ny);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    ctx->obst_epoch++;
    ctx->have_cost = true;
    ctx->ceff_dirty = true;
    return DYMU_OK;
}

int dymu_upload_terrain(dymu_ctx* ctx, const double* terrain, size_t ld)
{
    DYMU_GUARD(ctx);
    if (!ctx || !terrain || ld < ctx->nx) return DYMU_ERR_ARG;
    DYMU_TRY(ensure_stage(ctx));
    DYMU_CUDA_TRY(ctx, cudaMemcpy2DAsync(ctx->d_stage, ctx->nx * sizeof(double), terrain,
                                         ld * sizeof(double), ctx->nx * sizeof(double), ctx->ny,
                                         cudaMemcpyHostToDevice, ctx->stream));
    ctx->terrain_staged = true;
    return DYMU_OK;
}

int dymu_compute_cost_map(dymu_ctx* ctx, const double* cost_lut, int n_lut, const double* slopes,
                          int n_slopes, int n_locs, const double* elevation, size_t ld_e,
                          const double* terrain, size_t ld_t)
{
    DYMU_GUARD(ctx);
    if (!ctx || !cost_lut || !slopes || n_lut < 1 || n_slopes < 1 || n_locs < 1 || n_locs > 254)
        return DYMU_ERR_ARG;
    if (elevation)
    {
        if (ld_e < ctx->nx) return DYMU_ERR_ARG;
        DYMU_CUDA_TRY(ctx, cudaMemcpy2DAsync(ctx->elev, ctx->pitch * sizeof(double), elevation,
                                             ld_e * sizeof(double), ctx->nx * sizeof(double),
                                             ctx->ny, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (terrain) DYMU_TRY(dymu_upload_terrain(ctx, terrain, ld_t));
    if (!ctx->terrain_staged && !ctx->have_terrain)
        DYMU_FAIL(ctx, DYMU_ERR_STATE, "terrain map was never uploaded");
    const double* terrain_src = ctx->terrain_staged ? ctx->d_stage : nullptr;
    if (ctx->d_lut) cudaFree(ctx->d_lut);
    if (ctx->d_slopes) cudaFree(ctx->d_slopes);
    ctx->d_lut = ctx->d_slopes = nullptr;
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->d_lut, sizeof(double) * n_lut));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->d_slopes, sizeof(double) * n_slopes));
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_lut, cost_lut, sizeof(double) * n_lut,
                                       cudaMemcpyHostToDevice, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_slopes, slopes, sizeof(double) * n_slopes,
                                       cudaMemcpyHostToDevice, ctx->stream));
    ctx->n_lut = n_lut;
    ctx->n_slopes = n_slopes;
    ctx->n_locs = n_locs;
    double Cmax = cost_lut[0];  // std::max_element, G.cpp:221
    for (int q = 1; q < n_lut; ++q)
        if (cost_lut[q] > Cmax) Cmax = cost_lut[q];
    size_t n = (size_t)ctx->nx * ctx->ny;
    k_slope_nominal<<<stream_grid(ctx, n), kThreads, 0, ctx->stream>>>(
        ctx->elev, terrain_src, ctx->nx, ctx->d_lut, ctx->d_slopes, n_slopes, n_locs, n_lut, Cmax,
        ctx->gres, ctx->slope, ctx->raw, ctx->terrain, ctx->obst, ctx->locmode, ctx->traff,
        ctx->haz, ctx->pitch, ctx->nx, ctx->ny);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    k_smooth_cost<<<stream_grid(ctx, n), kThreads, 0, ctx->stream>>>(ctx->raw, ctx->cost,
                                                                    ctx->pitch, ctx->nx, ctx->ny);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));  // cost_lut/slopes are caller memory
    ctx->terrain_staged = false;
    ctx->have_terrain = true;
    ctx->obst_epoch++;
    ctx->have_cost = true;
    ctx->ceff_dirty = true;
    return DYMU_OK;
}

int dymu_time_stencils(dymu_ctx* ctx, float ms[6])
{
    DYMU_GUARD(ctx);
    if (!ctx || !ms) return DYMU_ERR_ARG;
    for (int k = 0; k < 6; ++k) ms[k] = -1.0f;
    size_t n = (size_t)ctx->nx * ctx->ny, np = (size_t)ctx->pitch * ctx->rows;
    DYMU_TRY(ensure_stage(ctx));
    ctx->terrain_staged = false;  // d_stage doubles as scratch below
    auto tick = [&](cudaEvent_t e) { return cudaEventRecord(e, ctx->stream); };
    auto lap = [&](int k) -> int {
        DYMU_CUDA_TRY(ctx, tick(ctx->ev1));
        DYMU_CUDA_TRY(ctx, cudaEventSynchronize(ctx->ev1));
        DYMU_CUDA_TRY(ctx, cudaEventElapsedTime(&ms[k], ctx->ev0, ctx->ev1));
        return DYMU_OK;
    };
    // warm-up + timed pass of each kernel; d_stage doubles as the scratch output
    for (int pass = 0; pass < 2; ++pass)
    {
        DYMU_CUDA_TRY(ctx, tick(ctx->ev0));
        k_fill_f64<<<stream_grid(ctx, n / 2 + 1), kThreads, 0, ctx->stream>>>(ctx->d_stage, 0.0, n);
        DYMU_TRY(lap(0));
        DYMU_CUDA_TRY(ctx, tick(ctx->ev0));
        k_ceff<<<stream_grid(ctx, np), kThreads, 0, ctx->stream>>>(ctx->cost, ctx->haz, ctx->traff, ctx->obst,
                                                                ctx->ceff, ctx->gres, ctx->pitch, ctx->rows,
                                                                ctx->nx, ctx->ny, nullptr);
        DYMU_TRY(lap(1));
        DYMU_CUDA_TRY(ctx, tick(ctx->ev0));
        k_readback<<<stream_grid(ctx, n), kThreads, 0, ctx->stream>>>(ctx->T, ctx->haz, ctx->traff, ctx->obst,
                                                                   ctx->d_stage, DYMU_XFORM_INF_TO_MINUS1,
                                                                   ctx->pitch, ctx->nx, ctx->ny);
        DYMU_TRY(lap(2));
        DYMU_CUDA_TRY(ctx, tick(ctx->ev0));
        k_set_cost_map<<<stream_grid(ctx, n), kThreads, 0, ctx->stream>>>(ctx->cost, ctx->obst, ctx->traff,
                                                                       ctx->haz, ctx->pitch, ctx->nx, ctx->ny);
        DYMU_TRY(lap(3));
        ctx->launches += 4;
    }
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    ctx->obst_epoch++;  // k_set_cost_map wrote the obstacle plane (with the values it already held)
    // k_ceff wrote the plain cost term: put the clearance-adjusted C_eff back (the band width stays)
    if (ctx->clear_on && !ctx->ceff_dirty) DYMU_TRY(dymu_internal_clearance_ceff(ctx, nullptr));
    return DYMU_OK;
}

int dymu_read_cells(dymu_ctx* ctx, int plane, uint32_t slot, const uint32_t* cell_index,
                    uint32_t n, double* out)
{
    DYMU_GUARD(ctx);
    if (!ctx || !cell_index || !out) return DYMU_ERR_ARG;
    if (n == 0) return DYMU_OK;
    if (plane == DYMU_PLANE_CLEARANCE) DYMU_TRY(dymu_internal_clearance_update(ctx));
    double* d = plane_ptr(ctx, plane);
    if (!d) return DYMU_ERR_ARG;
    if (plane == DYMU_PLANE_TOTAL_COST)
    {
        if (slot >= ctx->n_slots) return DYMU_ERR_ARG;
        d += (size_t)slot * ctx->pitch * ctx->rows;
    }
    for (uint32_t k = 0; k < n; ++k)
        if (cell_index[k] >= (uint64_t)ctx->nx * ctx->ny) return DYMU_ERR_ARG;
    DYMU_TRY(dymu_internal_scratch(ctx, (size_t)n * 12, (size_t)n * 12));
    uint32_t* d_idx = (uint32_t*)((char*)ctx->d_scratch + (size_t)n * 8);
    double* d_out = (double*)ctx->d_scratch;
    memcpy(ctx->h_pinned, cell_index, (size_t)n * 4);
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(d_idx, ctx->h_pinned, (size_t)n * 4, cudaMemcpyHostToDevice,
                                       ctx->stream));
    k_gather_cells<<<dymu_div_up(n, 128), 128, 0, ctx->stream>>>(d, ctx->pitch, ctx->nx, d_idx, n,
                                                                 d_out);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(out, d_out, (size_t)n * 8, cudaMemcpyDeviceToHost,
                                       ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DYMU_OK;
}

int dymu_read_node(dymu_ctx* ctx, uint32_t i, uint32_t j, double out[10])
{
    DYMU_GUARD(ctx);
    if (!ctx || !out || i >= ctx->nx || j >= ctx->ny) return DYMU_ERR_ARG;
    k_read_node<<<1, 1, 0, ctx->stream>>>(ctx->elev, ctx->slope, ctx->raw, ctx->cost, ctx->haz,
                                          ctx->traff, ctx->T, ctx->terrain, ctx->obst, ctx->locmode,
                                          (size_t)j * ctx->pitch + i, (double*)ctx->d_scratch);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(out, ctx->d_scratch, 10 * sizeof(double),
                                       cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DYMU_OK;
}

int dymu_set_anisotropy(dymu_ctx* ctx, const double* theta_deg, const double* factor, int n)
{
    DYMU_GUARD(ctx);
    if (!ctx || n < 0) return DYMU_ERR_ARG;
    if (n == 0)
    {
        if (ctx->aniso_n)
        {
            DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            cudaFree(ctx->dircost);
            ctx->dircost = nullptr;
            ctx->aniso_n = 0;
            ctx->solved = false;  // the resident map is not the isotropic fixed point
        }
        return DYMU_OK;
    }
    if (n < 2 || n > DYMU_ANISO_MAX || !theta_deg || !factor)
        DYMU_FAIL(ctx, DYMU_ERR_ARG, "anisotropy table: need 2..%d pairs", DYMU_ANISO_MAX);
    for (int k = 0; k < n; ++k)
    {
        if (!isfinite(theta_deg[k]) || !isfinite(factor[k]) || !(factor[k] > 0))
            DYMU_FAIL(ctx, DYMU_ERR_ARG, "anisotropy table: entry %d is not a finite angle with a finite factor > 0", k);
        if (k > 0 && !(theta_deg[k] > theta_deg[k - 1]))
            DYMU_FAIL(ctx, DYMU_ERR_ARG, "anisotropy table: angles must be strictly ascending (entry %d)", k);
    }
    if (!ctx->dircost)
        DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->dircost, 4 * (size_t)ctx->pitch * ctx->rows * sizeof(double)));
    for (int k = 0; k < n; ++k)
    {
        ctx->aniso_theta[k] = theta_deg[k];
        ctx->aniso_f[k] = factor[k];
    }
    ctx->aniso_n = n;
    ctx->solved = false;
    // a clean C_eff: build the planes now; otherwise the next refresh builds both
    if (!ctx->ceff_dirty) DYMU_TRY(build_dircost(ctx));
    return DYMU_OK;
}

int dymu_count_reached(dymu_ctx* ctx, uint32_t slot, uint64_t* n_finite)
{
    DYMU_GUARD(ctx);
    return dymu_count_leq(ctx, slot, 1.0 / 0.0, n_finite);
}

int dymu_count_leq(dymu_ctx* ctx, uint32_t slot, double threshold, uint64_t* n_finite)
{
    DYMU_GUARD(ctx);
    if (!ctx || !n_finite || slot >= ctx->n_slots) return DYMU_ERR_ARG;
    unsigned long long* d = (unsigned long long*)ctx->d_scratch;
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(d, 0, 8, ctx->stream));
    size_t n = (size_t)ctx->nx * ctx->ny;
    k_count_finite<<<stream_grid(ctx, n), kThreads, 0, ctx->stream>>>(
        ctx->T + (size_t)slot * ctx->pitch * ctx->rows, ctx->pitch, ctx->nx, ctx->ny, threshold, d);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    unsigned long long h = 0;
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(&h, d, 8, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *n_finite = h;
    return DYMU_OK;
}

}  // extern "C"

int dymu_internal_cost_rows(dymu_ctx* ctx, uint32_t j0, uint32_t j1)
{
    if (j0 >= j1 || j1 > ctx->ny) return DYMU_ERR_ARG;
    const size_t off = (size_t)j0 * ctx->pitch;
    const uint32_t nr = j1 - j0;
    const size_t n = (size_t)ctx->pitch * nr;
    k_set_cost_map<<<stream_grid(ctx, n), kThreads, 0, ctx->stream>>>(
        ctx->cost + off, ctx->obst + off, ctx->traff + off, ctx->haz + off, ctx->pitch, ctx->nx, nr);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    ctx->obst_epoch++;
    k_ceff<<<stream_grid(ctx, n), kThreads, 0, ctx->stream>>>(ctx->cost + off, ctx->haz + off, ctx->traff + off,
                                                             ctx->obst + off, ctx->ceff + off, ctx->gres,
                                                             ctx->pitch, nr, ctx->nx, nr, nullptr);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    return DYMU_OK;
}

int dymu_internal_settle_upload(dymu_ctx* ctx)
{
    if (!ctx->upload_pending) return DYMU_OK;
    ctx->upload_pending = false;
    DYMU_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_up, 0));
    size_t n = (size_t)ctx->nx * ctx->ny;
    k_set_cost_map<<<stream_grid(ctx, n), kThreads, 0, ctx->stream>>>(
        ctx->cost, ctx->obst, ctx->traff, ctx->haz, ctx->pitch, ctx->nx, ctx->ny);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    ctx->obst_epoch++;
    ctx->have_cost = true;
    ctx->ceff_dirty = true;
    return DYMU_OK;
}

int dymu_internal_band_from_rows(dymu_ctx* ctx, uint32_t j0, uint32_t j1)
{
    ctx->fim_band = 1.0 / 0.0;
    if (j0 >= j1 || j1 > ctx->rows) return DYMU_OK;
    const size_t n = (size_t)ctx->pitch * (j1 - j0);
    DYMU_TRY(dymu_internal_scratch(ctx, 64, 64));
    double* d = (double*)ctx->d_scratch;
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(d, 0, 16, ctx->stream));
    k_ceff_stats<<<stream_grid(ctx, n), kThreads, 0, ctx->stream>>>(ctx->ceff + (size_t)j0 * ctx->pitch, n, d);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    double h[2] = {0, 0};
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(h, d, 16, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (h[1] > 0) ctx->fim_band = kBandFactor * (double)kTile * (h[0] / h[1]);
    return DYMU_OK;
}

// the directional-cost planes from elevation, C_eff and the table, and the band width of the
// anisotropic solve (a few tile crossings worth of the mean directional cost)
static int build_dircost(dymu_ctx* ctx)
{
    const size_t n = (size_t)ctx->pitch * ctx->rows;
    AnisoTable tab;
    tab.n = ctx->aniso_n;
    for (int k = 0; k < DYMU_ANISO_MAX; ++k)
    {
        tab.theta[k] = k < tab.n ? ctx->aniso_theta[k] : 0.0;
        tab.f[k] = k < tab.n ? ctx->aniso_f[k] : 0.0;
    }
    DYMU_TRY(dymu_internal_scratch(ctx, 64, 64));
    double* d = (double*)ctx->d_scratch;
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(d, 0, 16, ctx->stream));
    k_dircost<<<stream_grid(ctx, n), kThreads, 0, ctx->stream>>>(ctx->elev, ctx->ceff, ctx->dircost, n, ctx->gres,
                                                                 ctx->pitch, ctx->rows, ctx->nx, ctx->ny, tab, d);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    double h[2] = {0, 0};
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(h, d, 16, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->aniso_band = h[1] > 0 ? kBandFactor * (double)kTile * (h[0] / h[1]) : 1.0 / 0.0;
    return DYMU_OK;
}

int dymu_internal_maps_factors(dymu_ctx* ctx)
{
    const size_t n = (size_t)ctx->pitch * ctx->rows;
    AnisoTable tab;
    tab.n = ctx->maniso_n;
    for (int k = 0; k < DYMU_ANISO_MAX; ++k)
    {
        tab.theta[k] = k < tab.n ? ctx->maniso_theta[k] : 0.0;
        tab.f[k] = k < tab.n ? ctx->maniso_f[k] : 0.0;
    }
    if (!ctx->maps_fac) DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->maps_fac, 4 * n * sizeof(double)));
    k_dirfactor<<<stream_grid(ctx, n), kThreads, 0, ctx->stream>>>(ctx->elev, ctx->maps_fac, n, ctx->gres, ctx->pitch,
                                                                   ctx->rows, ctx->nx, ctx->ny, tab);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    return DYMU_OK;
}

int dymu_internal_refresh_ceff(dymu_ctx* ctx)
{
    if (!ctx->ceff_dirty) return DYMU_OK;
    size_t n = (size_t)ctx->pitch * ctx->rows;
    // the same pass accumulates sum and count of the finite values: the band width of the tile
    // scheduler is a few tile crossings worth of total cost
    DYMU_TRY(dymu_internal_scratch(ctx, 64, 64));
    double* d = (double*)ctx->d_scratch;
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(d, 0, 16, ctx->stream));
    if (ctx->clear_on) DYMU_TRY(dymu_internal_clearance_ceff(ctx, d));
    else
    {
        k_ceff<<<stream_grid(ctx, n), kThreads, 0, ctx->stream>>>(ctx->cost, ctx->haz, ctx->traff,
                                                                 ctx->obst, ctx->ceff, ctx->gres,
                                                                 ctx->pitch, ctx->rows, ctx->nx,
                                                                 ctx->ny, d);
        ctx->launches++;
        DYMU_CUDA_TRY(ctx, cudaGetLastError());
    }
    double h[2] = {0, 0};
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(h, d, 16, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->fim_band = h[1] > 0 ? kBandFactor * (double)kTile * (h[0] / h[1]) : 1.0 / 0.0;
    ctx->ceff_dirty = false;
    if (ctx->aniso_n) DYMU_TRY(build_dircost(ctx));
    return DYMU_OK;
}
