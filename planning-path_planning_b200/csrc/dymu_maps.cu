// dymu_maps.cu -- batches of independent cost maps: map q has its own cost-term plane and is solved
// into total-cost slot q, many maps per launch of the tile solver (DESIGN.md section 12).
//
// A map is self-contained: its C_eff is what a freshly created context of the same size builds from
// dymu_set_cost_map(cost_q) (setCostMap, G.cpp:109-126, with the globalNode defaults hazard 0 and
// trafficability 1), whatever the context's own hazard, trafficability, obstacle and clearance state.
// k_map_ceff builds the planes in one streaming pass; the solve is k_fim's MODE 3 (MODE 0 reading
// the cost term of problem q at C + q * slot_stride) behind k_seed_maps, which tests each goal against
// its own plane.  The context's cost, obstacle, C_eff and export planes are never touched.
#include <stdlib.h>

#include "dymu_ctx.cuh"

namespace
{
constexpr int kMapThreads = 256;

// C_eff of maps [0, gridDim.y): plane q of dst from the ny x nx matrix at src + q * src_stride (row
// stride ld), +inf on obstacles (cost <= 0) and on the padding.  The same pass adds the sum and count of
// the finite values of map q to stats[2q], stats[2q+1] and sets bad[q] for a cell that is neither an
// obstacle nor finite (NaN, +inf, overflow).  8 B read + 8 B written per cell; src may be dst itself
// (host input, copied into the plane first: each thread reads the cell it writes).
__global__ void __launch_bounds__(kMapThreads) k_map_ceff(const double* src, size_t ld, size_t src_stride,
                                                          double* dst, size_t plane, uint32_t pitch, uint32_t rows,
                                                          uint32_t nx, uint32_t ny, double gres, double* stats,
                                                          uint32_t* bad)
{
    const uint32_t q = blockIdx.y;
    const double* s = src + (size_t)q * src_stride;
    double* d = dst + (size_t)q * plane;
    double sum = 0, cnt = 0;
    uint32_t invalid = 0;
    for (uint32_t j = blockIdx.x; j < rows; j += gridDim.x)
        for (uint32_t i = threadIdx.x; i < pitch; i += kMapThreads)
        {
            double c = DYMU_INF;
            if (i < nx && j < ny)
            {
                const double cost = s[(size_t)j * ld + i];
                if (!(cost <= 0))
                {
                    c = gres * cost * (2 + 0.0 - 1.0);  // k_ceff's expression, hazard 0, trafficability 1
                    if (c < DYMU_INF)
                    {
                        sum += c;
                        cnt += 1.0;
                    }
                    else
                        invalid = 1;
                }
            }
            d[(size_t)j * pitch + i] = c;
        }
    // one atomic per block and quantity: a map's blocks all add into the same two words
    __shared__ double s_sum[kMapThreads / 32], s_cnt[kMapThreads / 32];
    __shared__ uint32_t s_bad;
    if (threadIdx.x == 0) s_bad = 0;
    for (int o = 16; o > 0; o >>= 1)
    {
        sum += __shfl_down_sync(0xffffffffu, sum, o);
        cnt += __shfl_down_sync(0xffffffffu, cnt, o);
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0)
    {
        s_sum[threadIdx.x / 32] = sum;
        s_cnt[threadIdx.x / 32] = cnt;
    }
    if (invalid) s_bad = 1;
    __syncthreads();
    if (threadIdx.x == 0)
    {
        for (int w = 1; w < kMapThreads / 32; ++w)
        {
            sum += s_sum[w];
            cnt += s_cnt[w];
        }
        if (cnt > 0)
        {
            atomicAdd(&stats[2 * q], sum);
            atomicAdd(&stats[2 * q + 1], cnt);
        }
        if (s_bad) atomicOr(&bad[q], 1u);
    }
}

// device memory of the context's GPU (cudaMalloc'd or managed, e.g. a torch CUDA tensor)?
bool on_device(const dymu_ctx* ctx, const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess)
    {
        cudaGetLastError();
        return false;
    }
    return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) && a.device == ctx->device;
}
}  // namespace

int dymu_internal_fill(dymu_ctx* ctx, double* p, double v, size_t n);

void dymu_internal_maps_free(dymu_ctx* ctx)
{
    if (ctx->maps) cudaFree(ctx->maps);
    free(ctx->map_info);
    ctx->maps = nullptr;
    ctx->map_info = nullptr;
    ctx->n_maps = 0;
}

extern "C" {

int dymu_reserve_maps(dymu_ctx* ctx, uint32_t n_maps)
{
    DYMU_GUARD(ctx);
    if (!ctx) return DYMU_ERR_ARG;
    if (n_maps == ctx->n_maps) return DYMU_OK;
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    dymu_internal_maps_free(ctx);
    if (n_maps == 0) return DYMU_OK;
    if (ctx->n_slots < n_maps) DYMU_TRY(dymu_reserve_slots(ctx, n_maps));
    const size_t plane = (size_t)ctx->pitch * ctx->rows;
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->maps, plane * n_maps * sizeof(double)));
    ctx->map_info = (dymu_map_info*)calloc(n_maps, sizeof(dymu_map_info));
    if (!ctx->map_info)
    {
        dymu_internal_maps_free(ctx);
        DYMU_FAIL(ctx, DYMU_ERR_ARG, "dymu_reserve_maps: no host memory for %u maps", n_maps);
    }
    ctx->n_maps = n_maps;
    return DYMU_OK;
}

int dymu_set_maps(dymu_ctx* ctx, uint32_t first, uint32_t n, const double* cost, size_t ld, size_t map_stride,
                  int device_ptr)
{
    DYMU_GUARD(ctx);
    if (!ctx || !cost || ld < ctx->nx) return DYMU_ERR_ARG;
    if ((uint64_t)first + n > ctx->n_maps)
        DYMU_FAIL(ctx, DYMU_ERR_ARG, "maps [%u, %u) beyond the %u reserved (dymu_reserve_maps)", first,
                  first + n, ctx->n_maps);
    if (n == 0) return DYMU_OK;
    const size_t plane = (size_t)ctx->pitch * ctx->rows;
    double* dst = ctx->maps + (size_t)first * plane;
    const double* src = cost;
    size_t src_ld = ld, src_stride = map_stride;
    if (device_ptr)
    {
        const double* last = cost + (size_t)(n - 1) * map_stride + (size_t)(ctx->ny - 1) * ld + (ctx->nx - 1);
        if (!on_device(ctx, cost) || !on_device(ctx, last))
            DYMU_FAIL(ctx, DYMU_ERR_ARG, "dymu_set_maps: the matrices are not device memory of GPU %d", ctx->device);
    }
    else
    {
        // into the planes first, then transformed in place
        for (uint32_t q = 0; q < n; ++q)
            DYMU_CUDA_TRY(ctx, cudaMemcpy2DAsync(dst + (size_t)q * plane, ctx->pitch * sizeof(double),
                                                 cost + (size_t)q * map_stride, ld * sizeof(double),
                                                 ctx->nx * sizeof(double), ctx->ny, cudaMemcpyHostToDevice,
                                                 ctx->stream));
        src = dst;
        src_ld = ctx->pitch;
        src_stride = plane;
    }
    for (uint32_t q = 0; q < n; ++q) ctx->map_info[first + q].set = false;
    // per map: sum, count (doubles), then the invalid-value flags
    const size_t stat_bytes = (size_t)n * (2 * sizeof(double) + sizeof(uint32_t));
    DYMU_TRY(dymu_internal_scratch(ctx, stat_bytes, stat_bytes));
    double* d_stats = (double*)ctx->d_scratch;
    uint32_t* d_bad = (uint32_t*)(d_stats + 2 * (size_t)n);
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_scratch, 0, stat_bytes, ctx->stream));
    // a few waves of blocks over all maps; blockIdx.y = map (at most 65535 per launch)
    for (uint32_t q0 = 0; q0 < n; q0 += 65535u)
    {
        const uint32_t m = n - q0 < 65535u ? n - q0 : 65535u;
        uint32_t bx = (uint32_t)ctx->sm_count * 16u / m;
        bx = bx < 1u ? 1u : (bx > ctx->rows ? ctx->rows : bx);
        k_map_ceff<<<dim3(bx, m), kMapThreads, 0, ctx->stream>>>(
            src + (size_t)q0 * src_stride, src_ld, src_stride, dst + (size_t)q0 * plane, plane, ctx->pitch,
            ctx->rows, ctx->nx, ctx->ny, ctx->gres, d_stats + 2 * (size_t)q0, d_bad + q0);
        ctx->launches++;
        DYMU_CUDA_TRY(ctx, cudaGetLastError());
    }
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_pinned, ctx->d_scratch, stat_bytes, cudaMemcpyDeviceToHost,
                                       ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    const double* h_stats = (const double*)ctx->h_pinned;
    const uint32_t* h_bad = (const uint32_t*)(h_stats + 2 * (size_t)n);
    int64_t first_bad = -1;
    for (uint32_t q = 0; q < n; ++q)
    {
        if (h_bad[q])
        {
            if (first_bad < 0) first_bad = q;
            continue;
        }
        dymu_map_info& m = ctx->map_info[first + q];
        m.sum = h_stats[2 * q];
        m.count = h_stats[2 * q + 1];
        m.set = true;
    }
    if (first_bad >= 0)
        DYMU_FAIL(ctx, DYMU_ERR_ARG, "map %u holds a cost that is neither <= 0 nor gives a finite C_eff "
                  "(NaN, +inf or overflow); it is not set", first + (uint32_t)first_bad);
    return DYMU_OK;
}

int dymu_solve_maps(dymu_ctx* ctx, uint32_t n, const uint32_t* goal_i, const uint32_t* goal_j,
                    dymu_solve_stats* stats)
{
    DYMU_GUARD(ctx);
    if (!ctx || !goal_i || !goal_j || n < 1) return DYMU_ERR_ARG;
    if (n > ctx->n_maps || n > ctx->n_slots)
        DYMU_FAIL(ctx, DYMU_ERR_ARG, "%u maps: %u reserved (dymu_reserve_maps), %u total-cost slots", n, ctx->n_maps,
                  ctx->n_slots);
    for (uint32_t q = 0; q < n; ++q)
        if (goal_i[q] >= ctx->nx || goal_j[q] >= ctx->ny) DYMU_FAIL(ctx, DYMU_ERR_ARG, "goal %u outside the grid", q);
    if (ctx->aniso_n || ctx->clear_on)
        DYMU_FAIL(ctx, DYMU_ERR_STATE, "map batches are isotropic and without obstacle clearance");
    double sum = 0, count = 0;
    for (uint32_t q = 0; q < n; ++q)
    {
        if (!ctx->map_info[q].set) DYMU_FAIL(ctx, DYMU_ERR_STATE, "map %u was never set (dymu_set_maps)", q);
        sum += ctx->map_info[q].sum;
        count += ctx->map_info[q].count;
    }
    DYMU_TRY(dymu_internal_settle_delivery(ctx));
    // the slots are overwritten: slot 0 no longer holds the context's own solve nor a delivered matrix
    ctx->solved = false;
    ctx->export_done = false;
    const size_t plane = (size_t)ctx->pitch * ctx->rows;
    DYMU_CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    DYMU_TRY(dymu_internal_fill(ctx, ctx->T, 1.0 / 0.0, plane * n));
    DYMU_TRY(dymu_internal_scratch(ctx, (size_t)n * 8, (size_t)n * 8));
    uint32_t* h_goals = (uint32_t*)ctx->h_pinned;
    for (uint32_t q = 0; q < n; ++q)
    {
        h_goals[2 * q] = goal_i[q];
        h_goals[2 * q + 1] = goal_j[q];
    }
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_scratch, h_goals, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    dymu_fim_launch L;
    L.T = ctx->T; L.slot_stride = plane; L.C = ctx->maps;
    L.pitch = ctx->pitch; L.rows = ctx->rows; L.ntx = ctx->ntx; L.nty = ctx->nty; L.nprob = n;
    L.mode = 3;
    L.work = &ctx->work;
    // the band only orders work: one width for the launch, from the mean over all its maps
    L.band = count > 0 ? kBandFactor * (double)kTile * (sum / count) : 1.0 / 0.0;
    DYMU_TRY(dymu_internal_fim_seed_maps(ctx, &ctx->work, (const uint32_t*)ctx->d_scratch, n));
    dymu_solve_stats local;
    memset(&local, 0, sizeof(local));
    int rc = dymu_internal_fim_run(ctx, L, &local);
    if (rc == DYMU_OK || rc == DYMU_ERR_NOCONV)
    {
        cudaEventElapsedTime(&local.reset_ms, ctx->ev0, ctx->ev1);
        if (stats) *stats = local;
    }
    return rc;
}

}  // extern "C"
