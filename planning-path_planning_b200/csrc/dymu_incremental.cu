// dymu_incremental.cu -- re-solve of the total-cost map after the cost planes changed a little.
//
// The local layer feeds back into the global one: a repair lowers `trafficability` along the
// abandoned piece of path (L.cpp:388-394) and ingested obstacles raise `hazard_density`
// (L.cpp:264-274); both enter C = global_res * cost * (2 + hazard_density - trafficability)
// (G.cpp:527-528).  The reference answers with a full computeTotalCostMap.  Here only what can
// have changed is propagated again:
//
//   1. k_inc_diff   new C_eff for every cell, compared with the one the resident total-cost map
//                   was solved with.  A cell whose C went DOWN only needs its tile re-activated
//                   (values decrease monotonically, the solver absorbs that).  A cell whose C
//                   went UP carries a value that is now too small -- and so may every value
//                   computed from it.
//   2. k_inc_mark   breadth-first marking of that dependency cone: a reached cell depends at most
//                   on neighbours with a strictly smaller value (the update is upwind), so
//                   everything reachable from a raised cell along strictly increasing values is
//                   marked (a superset of the true cone: safe).  Unmarked cells keep values that
//                   are still exactly the fixed point of the new problem.
//   3. k_inc_apply  marked cells go back to +inf, their tiles are queued.
//   4. the tile FIM kernel runs from that seeded state.
//
// With obstacle clearance on, step 1 applies the clearance adjustment (dymu_clearance_ceff) to the
// resident clearance plane, rebuilt first if the obstacles changed.  The update stays monotone and
// upwind, so a cell whose adjusted C went up is a cone root like any other.
//
// The result is the fixed point of propagateGlobalNode (G.cpp:500-546) for the new planes, i.e.
// what a full solve gives, to rounding.  When the cone outgrows its buffer the call falls back to
// the full solve.
#include "dymu_ctx.cuh"

namespace
{
constexpr uint32_t kFullTile = 16u;  // activation flag "re-evaluate the whole tile" (dymu_fim.cu: kFull)

struct IncArgs
{
    const double *cost, *haz, *traff;
    const uint8_t* obst;
    double* ceff;
    double* T;
    uint32_t pitch, rows, nx, ny, ntx, tile_edge;  // tile_edge = kTile (the kernels take it at run time)
    double gres;
    uint32_t goal_cell_lo, goal_cell_hi;  // padded-plane index of the goal, split (kept out of the cone)
    uint32_t* markbits;                   // one bit per padded cell
    uint32_t* visited;                    // BFS queue == list of all marked cells
    uint32_t cap;
    uint32_t* counters;  // [0] queue tail, [1] overflow, [2] tiles woken for lowered cells, [3] marked total
    uint32_t* list0;
    uint32_t* flag0;
    unsigned long long* key0;
    unsigned long long* gmin;
    uint32_t* ctrl;
};

__device__ __forceinline__ void wake_tile(const IncArgs& a, size_t q)
{
    const uint32_t j = (uint32_t)(q / a.pitch), i = (uint32_t)(q % a.pitch);
    const uint32_t t = (j / a.tile_edge) * a.ntx + i / a.tile_edge;
    if (atomicOr(&a.flag0[t], kFullTile) == 0)
    {
        a.key0[t] = 0ull;
        a.list0[atomicAdd(&a.ctrl[kCtrlCount], 1u)] = t;
        a.gmin[0] = 0ull;
    }
}

// the clearance adjustment of k_inc_diff<true> (dymu_set_obstacle_clearance)
struct IncClear
{
    const double* clear;
    double radius, margin, penalty;
};

template <bool kClear>
__global__ void k_inc_diff(IncArgs a, IncClear cl)
{
    const size_t total = (size_t)a.pitch * a.rows;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t goal = ((size_t)a.goal_cell_hi << 32) | a.goal_cell_lo;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += stride)
    {
        const uint32_t j = (uint32_t)(q / a.pitch), i = (uint32_t)(q % a.pitch);
        double c = DYMU_INF;
        if (i < a.nx && j < a.ny && !a.obst[q])
        {
            c = a.gres * (a.cost[q]) * (2 + a.haz[q] - a.traff[q]);
            if (kClear) c = dymu_clearance_ceff(c, cl.clear[q], cl.radius, cl.margin, cl.penalty);
        }
        const double old = a.ceff[q];
        if (c == old) continue;
        a.ceff[q] = c;
        if (c < old)
        {
            wake_tile(a, q);
            atomicAdd(&a.counters[2], 1u);
        }
        else if (a.T[q] < DYMU_INF && q != goal)
        {
            // raised (or NaN-free "became an obstacle"): root of a dependency cone
            const uint32_t bit = 1u << (q & 31);
            if ((atomicOr(&a.markbits[q >> 5], bit) & bit) == 0)
            {
                const uint32_t pos = atomicAdd(&a.counters[0], 1u);
                if (pos < a.cap) a.visited[pos] = (uint32_t)q;
                else a.counters[1] = 1u;
            }
        }
    }
}

// level-synchronous breadth-first search by one CTA; the queue doubles as the list of marked cells
__global__ void __launch_bounds__(1024, 1) k_inc_mark(IncArgs a)
{
    __shared__ uint32_t s_head, s_tail;
    if (threadIdx.x == 0)
    {
        s_head = 0;
        s_tail = min(a.counters[0], a.cap);
    }
    __syncthreads();
    const size_t goal = ((size_t)a.goal_cell_hi << 32) | a.goal_cell_lo;
    for (;;)
    {
        const uint32_t head = s_head, tail = s_tail;
        if (head >= tail || *(volatile uint32_t*)&a.counters[1]) break;
        for (uint32_t k = head + threadIdx.x; k < tail; k += blockDim.x)
        {
            const uint32_t c = a.visited[k];
            const double tc = a.T[c];
            const uint32_t j = c / a.pitch, i = c % a.pitch;
            const int di[4] = {0, -1, 1, 0}, dj[4] = {-1, 0, 0, 1};
#pragma unroll
            for (int d = 0; d < 4; ++d)
            {
                const int ii = (int)i + di[d], jj = (int)j + dj[d];
                if (ii < 0 || jj < 0 || ii >= (int)a.nx || jj >= (int)a.ny) continue;
                const size_t q = (size_t)jj * a.pitch + ii;
                const double tn = a.T[q];
                if (!(tn > tc) || !(tn < DYMU_INF) || q == goal) continue;
                const uint32_t bit = 1u << (q & 31);
                if ((atomicOr(&a.markbits[q >> 5], bit) & bit) == 0)
                {
                    const uint32_t pos = atomicAdd(&a.counters[0], 1u);
                    if (pos < a.cap) a.visited[pos] = (uint32_t)q;
                    else a.counters[1] = 1u;
                }
            }
        }
        __threadfence_block();
        __syncthreads();
        if (threadIdx.x == 0)
        {
            s_head = tail;
            s_tail = min(*(volatile uint32_t*)&a.counters[0], a.cap);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) a.counters[3] = min(*(volatile uint32_t*)&a.counters[0], a.cap);
}

__global__ void k_inc_apply(IncArgs a, uint32_t n_marked)
{
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n_marked; k += stride)
    {
        const uint32_t c = a.visited[k];
        a.T[c] = DYMU_INF;
        wake_tile(a, c);
    }
}
}  // namespace

void dymu_internal_incremental_free(dymu_ctx* ctx)
{
    if (ctx->inc_markbits) cudaFree(ctx->inc_markbits);
    if (ctx->inc_visited) cudaFree(ctx->inc_visited);
    ctx->inc_markbits = ctx->inc_visited = nullptr;
    ctx->inc_cap = 0;
}

extern "C" {

int dymu_solve_incremental(dymu_ctx* ctx, uint32_t goal_i, uint32_t goal_j, dymu_solve_stats* stats,
                           uint64_t* cells_invalidated)
{
    DYMU_GUARD(ctx);
    if (!ctx || goal_i >= ctx->nx || goal_j >= ctx->ny) return DYMU_ERR_ARG;
    if (cells_invalidated) *cells_invalidated = UINT64_MAX;  // "everything": a full solve ran
    const size_t n = (size_t)ctx->pitch * ctx->rows;
    // the anisotropic solve has no invalidation cone: a change of C_eff or of the elevation moves
    // the directional costs of the cell and of its neighbours' pairs
    const bool reusable = !ctx->aniso_n && ctx->solved && ctx->last_n_goals == 1 && ctx->last_goal_i == goal_i
                          && ctx->last_goal_j == goal_j && !ctx->work.unclean && ctx->have_cost
                          && n < ((size_t)1 << 32);
    if (!reusable) return dymu_solve_total_cost(ctx, 1, &goal_i, &goal_j, stats);
    if (stats) memset(stats, 0, sizeof(*stats));
    // (an unchanged map keeps a matrix that was delivered directly; a partial re-solve does not)
    if (!ctx->ceff_dirty)
    {
        // nothing entered C_eff since the resident map was solved: it still is the answer
        if (stats) stats->converged = 1;
        if (cells_invalidated) *cells_invalidated = 0;
        return DYMU_OK;
    }
    if (!ctx->inc_markbits)
    {
        size_t cap = n / 4 < (1u << 16) ? (1u << 16) : n / 4;
        DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->inc_markbits, (n + 31) / 32 * sizeof(uint32_t)));
        DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->inc_visited, cap * sizeof(uint32_t)));
        ctx->inc_cap = (uint32_t)cap;
    }
    ctx->export_done = false;
    dymu_fim_work* w = &ctx->work;
    DYMU_TRY(dymu_internal_fim_clear(ctx, w));  // k_inc_diff / k_inc_apply queue the tiles
    DYMU_TRY(dymu_internal_clearance_update(ctx));  // the obstacles may have changed
    DYMU_TRY(dymu_internal_scratch(ctx, 64, 64));
    uint32_t* d_cnt = (uint32_t*)ctx->d_scratch;
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(d_cnt, 0, 16, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(ctx->inc_markbits, 0, (n + 31) / 32 * sizeof(uint32_t), ctx->stream));
    IncArgs a;
    a.cost = ctx->cost; a.haz = ctx->haz; a.traff = ctx->traff; a.obst = ctx->obst; a.ceff = ctx->ceff;
    a.T = ctx->T; a.pitch = ctx->pitch; a.rows = ctx->rows; a.nx = ctx->nx; a.ny = ctx->ny;
    a.ntx = ctx->ntx; a.tile_edge = kTile; a.gres = ctx->gres;
    const size_t goal = (size_t)goal_j * ctx->pitch + goal_i;
    a.goal_cell_lo = (uint32_t)goal; a.goal_cell_hi = (uint32_t)(goal >> 32);
    a.markbits = ctx->inc_markbits; a.visited = ctx->inc_visited; a.cap = ctx->inc_cap; a.counters = d_cnt;
    a.list0 = w->list[0]; a.flag0 = w->flag[0]; a.key0 = w->key[0]; a.gmin = w->gmin; a.ctrl = w->ctrl;
    int grid = (int)((n + 255) / 256);
    if (grid > ctx->sm_count * 16) grid = ctx->sm_count * 16;
    DYMU_CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    if (ctx->clear_on)
        k_inc_diff<true><<<grid, 256, 0, ctx->stream>>>(
            a, IncClear{ctx->clear, ctx->clear_radius, ctx->clear_margin, ctx->clear_penalty});
    else
        k_inc_diff<false><<<grid, 256, 0, ctx->stream>>>(a, IncClear{});
    k_inc_mark<<<1, 1024, 0, ctx->stream>>>(a);
    ctx->launches += 2;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    uint32_t h[4] = {0, 0, 0, 0};
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(h, d_cnt, 16, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->ceff_dirty = false;  // C_eff is up to date from here on
    if (h[1])
    {
        // the cone does not fit: nothing was invalidated yet, solve from scratch (the work lists
        // hold tiles woken for lowered cells: start clean)
        w->unclean = true;
        return dymu_solve_total_cost(ctx, 1, &goal_i, &goal_j, stats);
    }
    const uint32_t n_marked = h[3];
    if (cells_invalidated) *cells_invalidated = n_marked;
    if (n_marked == 0 && h[2] == 0)
    {
        if (stats) stats->converged = 1;  // only unreached cells changed their cost
        return DYMU_OK;
    }
    if (n_marked)
    {
        int g2 = (int)((n_marked + 255) / 256);
        if (g2 > ctx->sm_count * 8) g2 = ctx->sm_count * 8;
        k_inc_apply<<<g2, 256, 0, ctx->stream>>>(a, n_marked);
        ctx->launches++;
        DYMU_CUDA_TRY(ctx, cudaGetLastError());
    }
    dymu_solve_stats local;
    memset(&local, 0, sizeof(local));
    ctx->solved = false;
    int rc = dymu_internal_fim_run(ctx, dymu_internal_global_launch(ctx, 1), &local);
    if (rc == DYMU_OK || rc == DYMU_ERR_NOCONV)
    {
        cudaEventElapsedTime(&local.reset_ms, ctx->ev0, ctx->ev1);  // diff + marking + invalidation
        if (stats) *stats = local;
    }
    ctx->solved = (rc == DYMU_OK) && local.converged;
    return rc;
}

}  // extern "C"
