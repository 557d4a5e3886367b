// dymu_clearance.cu -- obstacle clearance of the total-cost solve (an extension; the reference plans
// for a point): the exact distance from every cell to the nearest obstacle cell within a window of
// R = floor((radius + margin) / global_res) cells, and C_eff with a lethal ring and a penalty margin
// around the obstacles (include/dymu_cuda.h, dymu_set_obstacle_clearance; DESIGN.md section 11).
//
// The squared distance s(i, j) = min over obstacles (i+di, j+dj), |di|, |dj| <= R, of di^2 + dj^2 is
// separable into two passes over the obstacle plane:
//   1. k_clear_cols   gcol(i, j) = min |dj| <= R to an obstacle in column i (u8 scratch plane; R <= 128)
//   2. k_clear_rows   s(i, j) = min over |di| <= R of di^2 + gcol(i+di, j)^2, from the row segment of
//                     the block and a halo of R cells in shared memory; writes the clearance plane and,
//                     fused, the clearance-adjusted C_eff
// When only cost, hazard or trafficability changed, k_ceff_clear rebuilds C_eff from the resident
// clearance plane.  Every solve reads C_eff (and the directional costs of slope anisotropy are built
// from it), so the tile solver and the path kernels need no change.
#include <limits.h>
#include <math.h>

#include "dymu_ctx.cuh"

namespace
{
constexpr uint8_t kNone = 255;        // gcol: no obstacle within R in the column
constexpr int kColThreads = 128;
constexpr int kColStrip = 256;        // rows per thread of the column pass
constexpr int kRowThreads = 256;      // columns per block of the row pass

struct ClearParams
{
    double gres, radius, margin, penalty, reach;  // reach = radius + margin
    int R;
};

// Column pass.  One thread per column and strip of kColStrip rows: a downward scan keeps the row of
// the last obstacle above, an upward scan the row of the next one below.  Consecutive threads read
// consecutive bytes of a row.  Per cell: (kColStrip + 2R) / kColStrip obstacle bytes read twice, gcol
// written twice and read once.  Cells outside the grid are not obstacles.
__global__ void __launch_bounds__(kColThreads) k_clear_cols(const uint8_t* __restrict__ obst,
                                                            uint8_t* __restrict__ gcol, uint32_t pitch,
                                                            uint32_t nx, uint32_t ny, int R)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const int j0 = (int)blockIdx.y * kColStrip;
    const int j1 = min(j0 + kColStrip, (int)ny);
    if (i >= pitch) return;
    if (i >= nx)
    {
        for (int j = j0; j < j1; ++j) gcol[(size_t)j * pitch + i] = kNone;
        return;
    }
    int last = INT_MIN / 2;
    for (int j = max(0, j0 - R); j < j1; ++j)
    {
        const size_t q = (size_t)j * pitch + i;
        if (obst[q]) last = j;
        if (j >= j0) gcol[q] = (j - last <= R) ? (uint8_t)(j - last) : kNone;
    }
    int next = INT_MAX / 2;
    for (int j = min((int)ny - 1, j1 - 1 + R); j >= j0; --j)
    {
        const size_t q = (size_t)j * pitch + i;
        if (obst[q]) next = j;
        if (j < j1 && next - j <= R)
        {
            const uint8_t g = gcol[q];
            if (next - j < g) gcol[q] = (uint8_t)(next - j);
        }
    }
}

// sum and count of the finite C_eff values of a block, one atomic pair per block
__device__ __forceinline__ void block_stats(double sum, double cnt, double* stats)
{
    __shared__ double s_sum[32], s_cnt[32];
    for (int o = 16; o > 0; o >>= 1)
    {
        sum += __shfl_down_sync(0xffffffffu, sum, o);
        cnt += __shfl_down_sync(0xffffffffu, cnt, o);
    }
    const int warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
    if ((threadIdx.x & 31) == 0)
    {
        s_sum[warp] = sum;
        s_cnt[warp] = cnt;
    }
    __syncthreads();
    if (threadIdx.x == 0)
    {
        double a = 0, b = 0;
        for (int w = 0; w < nwarps; ++w)
        {
            a += s_sum[w];
            b += s_cnt[w];
        }
        if (b > 0)
        {
            atomicAdd(&stats[0], a);
            atomicAdd(&stats[1], b);
        }
    }
}

// Row pass, fused with the C_eff build.  Block (x, y): columns [x * kRowThreads, +kRowThreads) of rows
// y, y + gridDim.y, ...; every padded cell is written (padding: +inf).  The candidates di are visited
// in increasing |di|: once di^2 reaches the best sum nothing farther can beat it.  Per cell: 1 B gcol
// (+ halo), and with `ceff` 25 B read + 8 B written; 8 B clearance written.
__global__ void __launch_bounds__(kRowThreads) k_clear_rows(const uint8_t* __restrict__ gcol,
                                                            const double* __restrict__ cost,
                                                            const double* __restrict__ haz,
                                                            const double* __restrict__ traff,
                                                            const uint8_t* __restrict__ obst,
                                                            double* __restrict__ clear, double* __restrict__ ceff,
                                                            ClearParams p, uint32_t pitch, uint32_t rows,
                                                            uint32_t nx, uint32_t ny, double* stats)
{
    __shared__ int s_g2[kRowThreads + 2 * DYMU_CLEARANCE_MAX_CELLS];  // gcol^2, -1: none
    const int R = p.R;
    const int i0 = (int)blockIdx.x * kRowThreads;
    const int t = (int)threadIdx.x, i = i0 + t;
    double sum = 0, cnt = 0;
    for (uint32_t j = blockIdx.y; j < rows; j += gridDim.y)
    {
        const bool in_row = j < ny;  // uniform over the block
        if (in_row)
        {
            __syncthreads();  // the previous row's readers are done
            for (int k = t; k < kRowThreads + 2 * R; k += kRowThreads)
            {
                const int ii = i0 - R + k;
                int v = -1;
                if (ii >= 0 && ii < (int)nx)
                {
                    const uint8_t g = gcol[(size_t)j * pitch + ii];
                    if (g != kNone) v = (int)g * (int)g;
                }
                s_g2[k] = v;
            }
            __syncthreads();
        }
        if (i >= (int)pitch) continue;
        const size_t q = (size_t)j * pitch + i;
        double d = DYMU_INF, c = DYMU_INF;
        if (in_row && i < (int)nx)
        {
            int best = INT_MAX;
            for (int k = 0; k <= R && k * k < best; ++k)
            {
                const int a = s_g2[R + t - k], b = s_g2[R + t + k];
                if (a >= 0) best = min(best, k * k + a);
                if (b >= 0) best = min(best, k * k + b);
            }
            if (best != INT_MAX)
            {
                const double e = sqrt((double)best) * p.gres;
                if (e <= p.reach) d = e;
            }
            if (ceff && !obst[q])
            {
                c = p.gres * (cost[q]) * (2 + haz[q] - traff[q]);
                c = dymu_clearance_ceff(c, d, p.radius, p.margin, p.penalty);
                if (c < DYMU_INF)
                {
                    sum += c;
                    cnt += 1.0;
                }
            }
        }
        clear[q] = d;
        if (ceff) ceff[q] = c;
    }
    if (stats) block_stats(sum, cnt, stats);
}

// C_eff from the resident clearance plane (cost, hazard or trafficability changed, the obstacles did
// not).  33 B read + 8 B written per cell.
__global__ void __launch_bounds__(256) k_ceff_clear(const double* __restrict__ cost, const double* __restrict__ haz,
                                                    const double* __restrict__ traff,
                                                    const uint8_t* __restrict__ obst,
                                                    const double* __restrict__ clear, double* __restrict__ ceff,
                                                    ClearParams p, uint32_t pitch, uint32_t rows, uint32_t nx,
                                                    uint32_t ny, double* stats)
{
    const size_t total = (size_t)pitch * rows;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    double sum = 0, cnt = 0;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += stride)
    {
        const uint32_t j = (uint32_t)(q / pitch), i = (uint32_t)(q % pitch);
        double c = DYMU_INF;
        if (i < nx && j < ny && !obst[q])
        {
            c = p.gres * (cost[q]) * (2 + haz[q] - traff[q]);
            c = dymu_clearance_ceff(c, clear[q], p.radius, p.margin, p.penalty);
            if (c < DYMU_INF)
            {
                sum += c;
                cnt += 1.0;
            }
        }
        ceff[q] = c;
    }
    if (stats) block_stats(sum, cnt, stats);
}

ClearParams params(const dymu_ctx* ctx)
{
    ClearParams p;
    p.gres = ctx->gres;
    p.radius = ctx->clear_radius;
    p.margin = ctx->clear_margin;
    p.penalty = ctx->clear_penalty;
    p.reach = ctx->clear_radius + ctx->clear_margin;
    p.R = (int)ctx->clear_R;
    return p;
}

bool fresh(const dymu_ctx* ctx) { return ctx->clear_fresh && ctx->clear_epoch == ctx->obst_epoch; }

// both passes; ceff == NULL: the clearance plane only
int build(dymu_ctx* ctx, double* ceff, double* stats)
{
    const dim3 gc(dymu_div_up(ctx->pitch, kColThreads), dymu_div_up(ctx->ny, kColStrip));
    k_clear_cols<<<gc, kColThreads, 0, ctx->stream>>>(ctx->obst, ctx->clear_gcol, ctx->pitch, ctx->nx, ctx->ny,
                                                     (int)ctx->clear_R);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    const uint32_t gx = dymu_div_up(ctx->pitch, kRowThreads);
    uint32_t gy = (uint32_t)ctx->sm_count * 16 / gx;
    gy = gy < 1 ? 1 : (gy > ctx->rows ? ctx->rows : gy);
    k_clear_rows<<<dim3(gx, gy), kRowThreads, 0, ctx->stream>>>(ctx->clear_gcol, ctx->cost, ctx->haz, ctx->traff,
                                                                ctx->obst, ctx->clear, ceff, params(ctx), ctx->pitch,
                                                                ctx->rows, ctx->nx, ctx->ny, stats);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    ctx->clear_fresh = true;
    ctx->clear_epoch = ctx->obst_epoch;
    return DYMU_OK;
}
}  // namespace

void dymu_internal_clearance_free(dymu_ctx* ctx)
{
    if (ctx->clear) cudaFree(ctx->clear);
    if (ctx->clear_gcol) cudaFree(ctx->clear_gcol);
    ctx->clear = nullptr;
    ctx->clear_gcol = nullptr;
    ctx->clear_on = ctx->clear_fresh = false;
}

int dymu_internal_clearance_update(dymu_ctx* ctx)
{
    if (!ctx->clear_on || fresh(ctx)) return DYMU_OK;
    return build(ctx, nullptr, nullptr);
}

int dymu_internal_clearance_ceff(dymu_ctx* ctx, double* stats)
{
    if (!fresh(ctx)) return build(ctx, ctx->ceff, stats);
    const size_t n = (size_t)ctx->pitch * ctx->rows;
    size_t blocks = (n + 255) / 256;
    if (blocks > (size_t)ctx->sm_count * 16) blocks = (size_t)ctx->sm_count * 16;
    k_ceff_clear<<<(unsigned)blocks, 256, 0, ctx->stream>>>(ctx->cost, ctx->haz, ctx->traff, ctx->obst, ctx->clear,
                                                           ctx->ceff, params(ctx), ctx->pitch, ctx->rows, ctx->nx,
                                                           ctx->ny, stats);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    return DYMU_OK;
}

extern "C" {

int dymu_set_obstacle_clearance(dymu_ctx* ctx, double radius, double margin, double penalty)
{
    DYMU_GUARD(ctx);
    if (!ctx) return DYMU_ERR_ARG;
    if (!isfinite(radius) || !isfinite(margin) || !isfinite(penalty) || radius < 0 || margin < 0 || penalty < 0)
        DYMU_FAIL(ctx, DYMU_ERR_ARG, "obstacle clearance: radius, margin and penalty must be finite and >= 0");
    if (radius == 0 && margin == 0)
    {
        if (ctx->clear_on)
        {
            DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            dymu_internal_clearance_free(ctx);
            ctx->ceff_dirty = true;
            ctx->solved = false;  // the resident map was solved with the adjusted costs
        }
        return DYMU_OK;
    }
    const double R = floor((radius + margin) / ctx->gres);
    if (!(R <= DYMU_CLEARANCE_MAX_CELLS))
        DYMU_FAIL(ctx, DYMU_ERR_ARG, "obstacle clearance: (radius + margin) / global_res = %g cells, at most %d",
                  R, DYMU_CLEARANCE_MAX_CELLS);
    const size_t n = (size_t)ctx->pitch * ctx->rows;
    if (!ctx->clear) DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->clear, n * sizeof(double)));
    if (!ctx->clear_gcol) DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->clear_gcol, n));
    ctx->clear_on = true;
    ctx->clear_fresh = false;
    ctx->clear_radius = radius;
    ctx->clear_margin = margin;
    ctx->clear_penalty = penalty;
    ctx->clear_R = (uint32_t)R;
    ctx->ceff_dirty = true;
    ctx->solved = false;
    return DYMU_OK;
}

}  // extern "C"
