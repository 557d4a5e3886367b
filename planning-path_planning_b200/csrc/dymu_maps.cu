// dymu_maps.cu -- batches of independent cost maps: map q has its own cost-term plane and is solved
// into total-cost slot q, many maps per launch of the tile solver (DESIGN.md section 12).
//
// A map is self-contained: its C_eff is what a freshly created context of the same size builds from
// dymu_set_cost_map(cost_q) (setCostMap, G.cpp:109-126, with the globalNode defaults hazard 0 and
// trafficability 1), whatever the context's own hazard, trafficability, obstacle and clearance state.
// k_map_ceff builds the planes in one streaming pass; the solve is k_fim's MODE 3 (MODE 0 reading
// the cost term of problem q at C + q * slot_stride) behind k_seed_maps, which tests each goal against
// its own plane.  The context's cost, obstacle, C_eff and export planes are never touched.
//
// Map batches have settings of their own (DESIGN.md section 13), apart from the context's:
//  - batch obstacle clearance (dymu_set_maps_clearance): the exact two-pass distance of
//    dymu_clearance.cu per map, batched over the maps (blockIdx.z = map): k_map_clear_cols on the
//    obstacles of map q (plain C_eff_q = +inf), k_map_clear_rows writing the adjusted C_eff_q into a
//    second set of planes (maps_adj) with the sum and count of its finite values.  The adjusted plane of
//    a map is rebuilt lazily, at the first solve after the map or the clearance changed.  The plain
//    planes stay the seeding planes.  The isotropic solve is MODE 3 on the adjusted planes.
//  - batch slope anisotropy (dymu_set_maps_anisotropy): four factor planes F_d = f(theta(x->m)) of the
//    context's elevation, shared by all maps (k_dirfactor, dymu_planes.cu), rebuilt at every solve;
//    the solve is MODE 4, which stages C_q(x) * F_d(x), and k_map_band sets its band.
#include <limits.h>
#include <math.h>
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

// ---- batch obstacle clearance: dymu_clearance.cu's two passes with the obstacles of map ids[z]
constexpr uint8_t kNone = 255;   // gcol: no obstacle within R in the column
constexpr int kColThreads = 128;
constexpr int kColStrip = 256;   // rows per thread of the column pass
constexpr int kRowThreads = 256; // columns per block of the row pass

struct MapClear
{
    double gres, radius, margin, penalty, reach;  // reach = radius + margin
    int R;
};

// k_clear_cols of map ids[blockIdx.z]: an obstacle is a cell of the grid whose plain C_eff is +inf
// (cost <= 0).  Per cell: (kColStrip + 2R) / kColStrip plain values read twice, gcol written twice, read once.
__global__ void __launch_bounds__(kColThreads) k_map_clear_cols(const double* __restrict__ maps,
                                                                const uint32_t* __restrict__ ids,
                                                                uint8_t* __restrict__ gcol, size_t plane,
                                                                uint32_t pitch, uint32_t nx, uint32_t ny, int R)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const int j0 = (int)blockIdx.y * kColStrip;
    const int j1 = min(j0 + kColStrip, (int)ny);
    if (i >= pitch) return;
    const size_t m = ids[blockIdx.z];
    const double* C = maps + m * plane;
    uint8_t* g = gcol + m * plane;
    if (i >= nx)
    {
        for (int j = j0; j < j1; ++j) g[(size_t)j * pitch + i] = kNone;
        return;
    }
    int last = INT_MIN / 2;
    for (int j = max(0, j0 - R); j < j1; ++j)
    {
        const size_t q = (size_t)j * pitch + i;
        if (!(C[q] < DYMU_INF)) last = j;
        if (j >= j0) g[q] = (j - last <= R) ? (uint8_t)(j - last) : kNone;
    }
    int next = INT_MAX / 2;
    for (int j = min((int)ny - 1, j1 - 1 + R); j >= j0; --j)
    {
        const size_t q = (size_t)j * pitch + i;
        if (!(C[q] < DYMU_INF)) next = j;
        if (j < j1 && next - j <= R)
        {
            const uint8_t v = g[q];
            if (next - j < v) g[q] = (uint8_t)(next - j);
        }
    }
}

// k_clear_rows of map ids[blockIdx.z], writing only the adjusted C_eff: +inf on the obstacles and the
// padding, dymu_clearance_ceff(plain C_eff, d) elsewhere -- the solo context's C_eff bit for bit, since
// the plain C_eff_q is its g * cost * (2 + hazard - trafficability).  The sum and count of the finite
// values go to stats[2z], stats[2z+1].  Per cell: 1 B gcol (+ halo), 8 B read, 8 B written.
__global__ void __launch_bounds__(kRowThreads) k_map_clear_rows(const uint8_t* __restrict__ gcol,
                                                                const double* __restrict__ maps,
                                                                const uint32_t* __restrict__ ids,
                                                                double* __restrict__ adj, size_t plane,
                                                                MapClear p, uint32_t pitch, uint32_t rows,
                                                                uint32_t nx, uint32_t ny, double* stats)
{
    __shared__ int s_g2[kRowThreads + 2 * DYMU_CLEARANCE_MAX_CELLS];  // gcol^2, -1: none
    const size_t m = ids[blockIdx.z];
    const uint8_t* g = gcol + m * plane;
    const double* C = maps + m * plane;
    double* A = adj + m * plane;
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
                    const uint8_t gv = g[(size_t)j * pitch + ii];
                    if (gv != kNone) v = (int)gv * (int)gv;
                }
                s_g2[k] = v;
            }
            __syncthreads();
        }
        if (i >= (int)pitch) continue;
        const size_t q = (size_t)j * pitch + i;
        double c = DYMU_INF;
        if (in_row && i < (int)nx)
        {
            const double plain = C[q];
            if (plain < DYMU_INF)
            {
                int best = INT_MAX;
                for (int k = 0; k <= R && k * k < best; ++k)
                {
                    const int a = s_g2[R + t - k], b = s_g2[R + t + k];
                    if (a >= 0) best = min(best, k * k + a);
                    if (b >= 0) best = min(best, k * k + b);
                }
                double d = DYMU_INF;
                if (best != INT_MAX)
                {
                    const double e = sqrt((double)best) * p.gres;
                    if (e <= p.reach) d = e;
                }
                c = dymu_clearance_ceff(plain, d, p.radius, p.margin, p.penalty);
                if (c < DYMU_INF)
                {
                    sum += c;
                    cnt += 1.0;
                }
            }
        }
        A[q] = c;
    }
    __shared__ double s_sum[kRowThreads / 32], s_cnt[kRowThreads / 32];
    for (int o = 16; o > 0; o >>= 1)
    {
        sum += __shfl_down_sync(0xffffffffu, sum, o);
        cnt += __shfl_down_sync(0xffffffffu, cnt, o);
    }
    if ((threadIdx.x & 31) == 0)
    {
        s_sum[threadIdx.x / 32] = sum;
        s_cnt[threadIdx.x / 32] = cnt;
    }
    __syncthreads();
    if (threadIdx.x == 0)
    {
        for (int w = 1; w < kRowThreads / 32; ++w)
        {
            sum += s_sum[w];
            cnt += s_cnt[w];
        }
        if (cnt > 0)
        {
            atomicAdd(&stats[2 * blockIdx.z], sum);
            atomicAdd(&stats[2 * blockIdx.z + 1], cnt);
        }
    }
}

// Band of an anisotropic map launch: sum and count of the finite directional costs C_q(x) * F_d(x) of
// maps [0, gridDim.y) into stats[0..1] (the band only orders work).  8 B of C_q read per cell and
// map, the factor planes (32 B per cell) once per map, mostly from L2.
__global__ void __launch_bounds__(kMapThreads) k_map_band(const double* __restrict__ C,
                                                          const double* __restrict__ F, size_t plane,
                                                          double* stats)
{
    const double* c = C + (size_t)blockIdx.y * plane;
    const size_t stride = (size_t)gridDim.x * kMapThreads;
    double sum = 0, cnt = 0;
    for (size_t q = (size_t)blockIdx.x * kMapThreads + threadIdx.x; q < plane; q += stride)
    {
        const double cq = c[q];
        if (!(cq < DYMU_INF)) continue;
#pragma unroll
        for (int d = 0; d < 4; ++d)
        {
            const double a = cq * F[d * plane + q];
            if (a < DYMU_INF)
            {
                sum += a;
                cnt += 1.0;
            }
        }
    }
    __shared__ double s_sum[kMapThreads / 32], s_cnt[kMapThreads / 32];
    for (int o = 16; o > 0; o >>= 1)
    {
        sum += __shfl_down_sync(0xffffffffu, sum, o);
        cnt += __shfl_down_sync(0xffffffffu, cnt, o);
    }
    if ((threadIdx.x & 31) == 0)
    {
        s_sum[threadIdx.x / 32] = sum;
        s_cnt[threadIdx.x / 32] = cnt;
    }
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
            atomicAdd(&stats[0], sum);
            atomicAdd(&stats[1], cnt);
        }
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

namespace
{
void free_clearance_planes(dymu_ctx* ctx)
{
    if (ctx->maps_adj) cudaFree(ctx->maps_adj);
    if (ctx->maps_gcol) cudaFree(ctx->maps_gcol);
    ctx->maps_adj = nullptr;
    ctx->maps_gcol = nullptr;
    for (uint32_t q = 0; q < ctx->n_maps; ++q) ctx->map_info[q].adj_fresh = false;
}

// slots [first, first + n) written by an anisotropic map solve no longer match its planes
void stale_marks(dymu_ctx* ctx, uint32_t first, uint32_t n)
{
    if (!ctx->slot_mark) return;
    for (uint32_t s = first; s < first + n && s < ctx->n_slots; ++s)
        if (ctx->slot_mark[s] == kSlotMapAniso) ctx->slot_mark[s] = kSlotMapAnisoStale;
}

MapClear clear_params(const dymu_ctx* ctx)
{
    MapClear p;
    p.gres = ctx->gres;
    p.radius = ctx->mclear_radius;
    p.margin = ctx->mclear_margin;
    p.penalty = ctx->mclear_penalty;
    p.reach = ctx->mclear_radius + ctx->mclear_margin;
    p.R = (int)ctx->mclear_R;
    return p;
}

// the adjusted C_eff of every stale map among [0, n): both passes, batched over those maps
int rebuild_adjusted(dymu_ctx* ctx, uint32_t n)
{
    const size_t plane = (size_t)ctx->pitch * ctx->rows;
    if (!ctx->maps_adj) DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->maps_adj, plane * ctx->n_maps * sizeof(double)));
    if (!ctx->maps_gcol) DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->maps_gcol, plane * ctx->n_maps));
    uint32_t m = 0;
    for (uint32_t q = 0; q < n; ++q) m += ctx->map_info[q].adj_fresh ? 0u : 1u;
    if (m == 0) return DYMU_OK;
    // per stale map: sum, count (doubles), then the map indices
    const size_t stat_bytes = (size_t)m * 2 * sizeof(double), bytes = stat_bytes + (size_t)m * sizeof(uint32_t);
    DYMU_TRY(dymu_internal_scratch(ctx, bytes, bytes));
    uint32_t* h_ids = (uint32_t*)((char*)ctx->h_pinned + stat_bytes);
    for (uint32_t q = 0, k = 0; q < n; ++q)
        if (!ctx->map_info[q].adj_fresh) h_ids[k++] = q;
    double* d_stats = (double*)ctx->d_scratch;
    const uint32_t* d_ids = (const uint32_t*)((char*)ctx->d_scratch + stat_bytes);
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(d_stats, 0, stat_bytes, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync((void*)d_ids, h_ids, (size_t)m * sizeof(uint32_t), cudaMemcpyHostToDevice,
                                       ctx->stream));
    const MapClear p = clear_params(ctx);
    for (uint32_t k0 = 0; k0 < m; k0 += 65535u)
    {
        const uint32_t mz = m - k0 < 65535u ? m - k0 : 65535u;
        const dim3 gc(dymu_div_up(ctx->pitch, kColThreads), dymu_div_up(ctx->ny, kColStrip), mz);
        k_map_clear_cols<<<gc, kColThreads, 0, ctx->stream>>>(ctx->maps, d_ids + k0, ctx->maps_gcol, plane,
                                                             ctx->pitch, ctx->nx, ctx->ny, p.R);
        ctx->launches++;
        DYMU_CUDA_TRY(ctx, cudaGetLastError());
        // a few waves of blocks over all maps of the launch
        const uint32_t gx = dymu_div_up(ctx->pitch, kRowThreads);
        uint32_t gy = (uint32_t)ctx->sm_count * 16u / (gx * mz);
        gy = gy < 1u ? 1u : (gy > ctx->rows ? ctx->rows : gy);
        k_map_clear_rows<<<dim3(gx, gy, mz), kRowThreads, 0, ctx->stream>>>(
            ctx->maps_gcol, ctx->maps, d_ids + k0, ctx->maps_adj, plane, p, ctx->pitch, ctx->rows, ctx->nx,
            ctx->ny, d_stats + 2 * (size_t)k0);
        ctx->launches++;
        DYMU_CUDA_TRY(ctx, cudaGetLastError());
    }
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_pinned, d_stats, stat_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    const double* h_stats = (const double*)ctx->h_pinned;
    for (uint32_t k = 0; k < m; ++k)
    {
        dymu_map_info& mi = ctx->map_info[h_ids[k]];
        mi.adj_sum = h_stats[2 * k];
        mi.adj_count = h_stats[2 * k + 1];
        mi.adj_fresh = true;
    }
    return DYMU_OK;
}

// band width of an anisotropic launch over maps [0, n) of the cost-term planes C
int aniso_band(dymu_ctx* ctx, const double* C, uint32_t n, double* band)
{
    const size_t plane = (size_t)ctx->pitch * ctx->rows;
    DYMU_TRY(dymu_internal_scratch(ctx, 64, 64));
    double* d = (double*)ctx->d_scratch;
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(d, 0, 16, ctx->stream));
    for (uint32_t q0 = 0; q0 < n; q0 += 65535u)
    {
        const uint32_t m = n - q0 < 65535u ? n - q0 : 65535u;
        uint32_t bx = (uint32_t)ctx->sm_count * 16u / m;
        const uint32_t bmax = (uint32_t)((plane + kMapThreads - 1) / kMapThreads);
        bx = bx < 1u ? 1u : (bx > bmax ? bmax : bx);
        k_map_band<<<dim3(bx, m), kMapThreads, 0, ctx->stream>>>(C + (size_t)q0 * plane, ctx->maps_fac, plane, d);
        ctx->launches++;
        DYMU_CUDA_TRY(ctx, cudaGetLastError());
    }
    double h[2] = {0, 0};
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(h, d, 16, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *band = h[1] > 0 ? kBandFactor * (double)kTile * (h[0] / h[1]) : 1.0 / 0.0;
    return DYMU_OK;
}
}  // namespace

void dymu_internal_maps_free(dymu_ctx* ctx)
{
    if (ctx->map_info) free_clearance_planes(ctx);
    if (ctx->maps_fac) cudaFree(ctx->maps_fac);
    ctx->maps_fac = nullptr;
    if (ctx->maps) cudaFree(ctx->maps);
    free(ctx->map_info);
    ctx->maps = nullptr;
    ctx->map_info = nullptr;
    ctx->n_maps = 0;
}

void dymu_internal_unmark_slots(dymu_ctx* ctx, uint32_t first, uint32_t n)
{
    if (!ctx->slot_mark) return;
    for (uint32_t s = first; s < first + n && s < ctx->n_slots; ++s) ctx->slot_mark[s] = kSlotPlain;
}

void dymu_internal_unmark_all(dymu_ctx* ctx)
{
    free(ctx->slot_mark);
    ctx->slot_mark = nullptr;
}

extern "C" {

int dymu_reserve_maps(dymu_ctx* ctx, uint32_t n_maps)
{
    DYMU_GUARD(ctx);
    if (!ctx) return DYMU_ERR_ARG;
    if (n_maps == ctx->n_maps) return DYMU_OK;
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    stale_marks(ctx, 0, ctx->n_slots);
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
    for (uint32_t q = 0; q < n; ++q) ctx->map_info[first + q].set = ctx->map_info[first + q].adj_fresh = false;
    stale_marks(ctx, first, n);
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
    for (uint32_t q = 0; q < n; ++q)
        if (!ctx->map_info[q].set) DYMU_FAIL(ctx, DYMU_ERR_STATE, "map %u was never set (dymu_set_maps)", q);
    DYMU_TRY(dymu_internal_settle_delivery(ctx));
    // the cost term of the solve: the plain planes, or the clearance-adjusted ones (seeding always
    // tests the plain planes: a goal inside the lethal ring is seeded, as in dymu_solve_total_cost)
    const double* C = ctx->maps;
    if (ctx->mclear_on)
    {
        DYMU_TRY(rebuild_adjusted(ctx, n));
        C = ctx->maps_adj;
    }
    double sum = 0, count = 0;
    for (uint32_t q = 0; q < n; ++q)
    {
        sum += ctx->mclear_on ? ctx->map_info[q].adj_sum : ctx->map_info[q].sum;
        count += ctx->mclear_on ? ctx->map_info[q].adj_count : ctx->map_info[q].count;
    }
    // the band only orders work: one width for the launch, from the mean over all its maps
    double band = count > 0 ? kBandFactor * (double)kTile * (sum / count) : 1.0 / 0.0;
    if (ctx->maniso_n)
    {
        DYMU_TRY(dymu_internal_maps_factors(ctx));
        DYMU_TRY(aniso_band(ctx, C, n, &band));
        if (!ctx->slot_mark)
        {
            ctx->slot_mark = (uint8_t*)calloc(ctx->n_slots, 1);
            if (!ctx->slot_mark) DYMU_FAIL(ctx, DYMU_ERR_ARG, "dymu_solve_maps: no host memory for the slot marks");
        }
        // the factor planes were rebuilt from the elevation as it is now: older anisotropic map slots
        // beyond this launch may no longer match them
        stale_marks(ctx, n, ctx->n_slots - n);
        memset(ctx->slot_mark, kSlotMapAniso, n);
    }
    else
        dymu_internal_unmark_slots(ctx, 0, n);
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
    L.T = ctx->T; L.slot_stride = plane; L.C = C;
    L.pitch = ctx->pitch; L.rows = ctx->rows; L.ntx = ctx->ntx; L.nty = ctx->nty; L.nprob = n;
    L.mode = ctx->maniso_n ? 4 : 3;
    L.A = ctx->maniso_n ? ctx->maps_fac : nullptr;
    L.work = &ctx->work;
    L.band = band;
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

int dymu_set_maps_clearance(dymu_ctx* ctx, double radius, double margin, double penalty)
{
    DYMU_GUARD(ctx);
    if (!ctx) return DYMU_ERR_ARG;
    if (!isfinite(radius) || !isfinite(margin) || !isfinite(penalty) || radius < 0 || margin < 0 || penalty < 0)
        DYMU_FAIL(ctx, DYMU_ERR_ARG, "obstacle clearance: radius, margin and penalty must be finite and >= 0");
    if (radius == 0 && margin == 0)
    {
        if (ctx->mclear_on)
        {
            DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            free_clearance_planes(ctx);
            ctx->mclear_on = false;
            stale_marks(ctx, 0, ctx->n_slots);
        }
        return DYMU_OK;
    }
    const double R = floor((radius + margin) / ctx->gres);
    if (!(R <= DYMU_CLEARANCE_MAX_CELLS))
        DYMU_FAIL(ctx, DYMU_ERR_ARG, "obstacle clearance: (radius + margin) / global_res = %g cells, at most %d",
                  R, DYMU_CLEARANCE_MAX_CELLS);
    if (ctx->mclear_on && ctx->mclear_radius == radius && ctx->mclear_margin == margin
        && ctx->mclear_penalty == penalty)
        return DYMU_OK;
    ctx->mclear_on = true;
    ctx->mclear_radius = radius;
    ctx->mclear_margin = margin;
    ctx->mclear_penalty = penalty;
    ctx->mclear_R = (uint32_t)R;
    for (uint32_t q = 0; q < ctx->n_maps; ++q) ctx->map_info[q].adj_fresh = false;
    stale_marks(ctx, 0, ctx->n_slots);
    return DYMU_OK;
}

int dymu_set_maps_anisotropy(dymu_ctx* ctx, const double* theta_deg, const double* factor, int n)
{
    DYMU_GUARD(ctx);
    if (!ctx || n < 0) return DYMU_ERR_ARG;
    if (n == 0)
    {
        if (ctx->maniso_n)
        {
            DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            if (ctx->maps_fac) cudaFree(ctx->maps_fac);
            ctx->maps_fac = nullptr;
            ctx->maniso_n = 0;
            stale_marks(ctx, 0, ctx->n_slots);
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
    bool same = ctx->maniso_n == n;
    for (int k = 0; k < n && same; ++k) same = ctx->maniso_theta[k] == theta_deg[k] && ctx->maniso_f[k] == factor[k];
    if (same) return DYMU_OK;
    for (int k = 0; k < n; ++k)
    {
        ctx->maniso_theta[k] = theta_deg[k];
        ctx->maniso_f[k] = factor[k];
    }
    ctx->maniso_n = n;
    stale_marks(ctx, 0, ctx->n_slots);
    return DYMU_OK;
}

}  // extern "C"
