// dymu_multi.cu -- several contexts (one per GPU) driven from one call: the two cases of
// SURVEY.md section 8(e) in which DyMu's total-cost propagation shards.
//
//   dymu_batch_solve  independent goal queries on copies of one cost map: the queries are dealt
//                     out in contiguous blocks, one host thread per context, no data-path
//                     exchange at all (the reference would run one planner instance per query:
//                     computeEntireTotalCostMap G.cpp:443-468 + getPath G.cpp:589-611).
//   dymu_dd_solve     ONE grid cut into row strips, one strip per context.  A strip carries one
//                     ghost row per interior side whose cost is 0 (obstacle: never a propagation
//                     target), so it acts as Dirichlet data.  Every round each strip advances by
//                     a bounded number of solver phases, then its first / last own row goes
//                     straight into the neighbour's inbox on the neighbour's GPU
//                     (cudaMemcpyPeerAsync over NVLink), the neighbour min-merges it into its
//                     ghost row and re-activates the tiles along it.  Values only ever decrease,
//                     so the strips converge to the single-grid fixed point.  Synchronisation per
//                     round: the two stream synchronisations inside the solver calls of each strip
//                     and one host barrier between the strip threads -- no device-wide
//                     synchronisation, no host round trip of the rows.
#include <pthread.h>
#include <time.h>

#include <vector>

#include "dymu_ctx.cuh"

namespace
{
double now_ms()
{
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}

struct DdShared
{
    dymu_ctx** ctxs;
    uint32_t n;
    const uint32_t* cuts;  // n + 1 global rows: strip k owns [cuts[k], cuts[k + 1])
    uint32_t goal_i, goal_j, phases, max_rounds;
    pthread_barrier_t bar;
    std::vector<double*> inbox;        // per strip: 2 rows on its own device ([0] from above, [1] from below)
    std::vector<cudaEvent_t> sent;     // per strip: its exports of this round are enqueued
    std::vector<int> busy;             // per strip: pending work or fresh halo values this round
    std::vector<int> rc;
    std::vector<float> kernel_ms;
    std::vector<unsigned long long> activations, updates;
    uint32_t rounds;
    int any_failed;
};

struct DdThread
{
    DdShared* s;
    uint32_t k;
};

void* dd_worker(void* arg)
{
    DdThread* t = (DdThread*)arg;
    DdShared& S = *t->s;
    const uint32_t k = t->k, n = S.n;
    dymu_ctx* ctx = S.ctxs[k];
    dymu_device_guard guard(ctx->device);
    const uint32_t ghost_top = k > 0 ? 1u : 0u;
    const uint32_t own = S.cuts[k + 1] - S.cuts[k];
    const uint32_t first_own = ghost_top, last_own = ghost_top + own - 1;
    const uint32_t ny_local = own + ghost_top + (k + 1 < n ? 1u : 0u);
    const size_t row_bytes = (size_t)ctx->nx * sizeof(double);
    int rc = DYMU_OK;
    bool pending = false;
    dymu_solve_stats st;
    auto account = [&](const dymu_solve_stats& q) {
        S.kernel_ms[k] += q.kernel_ms;
        S.activations[k] += q.tile_activations;
        S.updates[k] += q.cell_updates;
    };
    // round 0: the strip that owns the goal seeds it, the others start from +inf
    if (S.goal_j >= S.cuts[k] && S.goal_j < S.cuts[k + 1])
    {
        memset(&st, 0, sizeof(st));
        rc = dymu_solve_start(ctx, S.goal_i, S.goal_j - S.cuts[k] + ghost_top, S.phases, &st);
        if (rc == DYMU_OK)
        {
            pending = !st.converged;
            account(st);
        }
    }
    else
        rc = dymu_reset_total_cost(ctx);
    uint32_t round = 0;
    for (;;)
    {
        // ---- my boundary rows go into the neighbours' inboxes, on my stream
        if (rc == DYMU_OK && k > 0)
        {
            const double* src = ctx->T + (size_t)first_own * ctx->pitch;
            cudaError_t e = cudaMemcpyPeerAsync(S.inbox[k - 1] + ctx->nx, S.ctxs[k - 1]->device, src, ctx->device,
                                                row_bytes, ctx->stream);
            if (e != cudaSuccess) rc = DYMU_ERR_CUDA;
        }
        if (rc == DYMU_OK && k + 1 < n)
        {
            const double* src = ctx->T + (size_t)last_own * ctx->pitch;
            cudaError_t e = cudaMemcpyPeerAsync(S.inbox[k + 1], S.ctxs[k + 1]->device, src, ctx->device, row_bytes,
                                                ctx->stream);
            if (e != cudaSuccess) rc = DYMU_ERR_CUDA;
        }
        if (cudaEventRecord(S.sent[k], ctx->stream) != cudaSuccess) rc = DYMU_ERR_CUDA;
        if (rc != DYMU_OK) S.any_failed = 1;
        pthread_barrier_wait(&S.bar);  // every strip has enqueued its exports
        if (S.any_failed) break;
        // ---- min-merge what the neighbours sent into my ghost rows
        uint32_t ranges[4], n_ranges = 0;
        double key = 1.0 / 0.0;
        if (k > 0)
        {
            int changed = 0;
            double lo = 0;
            if (cudaStreamWaitEvent(ctx->stream, S.sent[k - 1], 0) != cudaSuccess) rc = DYMU_ERR_CUDA;
            if (rc == DYMU_OK) rc = dymu_import_rows_min_key(ctx, 0, 0, 1, S.inbox[k], 1, &changed, &lo);
            if (rc == DYMU_OK && changed)
            {
                ranges[2 * n_ranges] = 0;
                ranges[2 * n_ranges + 1] = 2;
                n_ranges++;
                if (lo < key) key = lo;
            }
        }
        if (k + 1 < n)
        {
            int changed = 0;
            double lo = 0;
            if (cudaStreamWaitEvent(ctx->stream, S.sent[k + 1], 0) != cudaSuccess) rc = DYMU_ERR_CUDA;
            if (rc == DYMU_OK)
                rc = dymu_import_rows_min_key(ctx, 0, ny_local - 1, 1, S.inbox[k] + ctx->nx, 1, &changed, &lo);
            if (rc == DYMU_OK && changed)
            {
                ranges[2 * n_ranges] = ny_local - 2;
                ranges[2 * n_ranges + 1] = ny_local;
                n_ranges++;
                if (lo < key) key = lo;
            }
        }
        S.busy[k] = (pending || n_ranges > 0) ? 1 : 0;
        if (rc != DYMU_OK) S.any_failed = 1;
        pthread_barrier_wait(&S.bar);  // votes are in; the inboxes have been consumed
        if (S.any_failed) break;
        bool any = false;
        for (uint32_t q = 0; q < n; ++q) any = any || S.busy[q];
        round++;
        if (!any || round >= S.max_rounds) break;
        // ---- bounded advance; re-activated halo tiles enter the band with the smallest
        // imported value as their key
        if (pending || n_ranges > 0)
        {
            memset(&st, 0, sizeof(st));
            rc = dymu_solve_advance(ctx, ranges, n_ranges, n_ranges ? key : 0.0, S.phases, &st);
            if (rc == DYMU_OK)
            {
                pending = !st.converged;
                account(st);
            }
        }
    }
    if (k == 0) S.rounds = round;
    S.rc[k] = rc;
    if (rc == DYMU_OK && pending) S.rc[k] = DYMU_ERR_NOCONV;
    ctx->solved = (S.rc[k] == DYMU_OK);
    return nullptr;
}

struct BatchShared
{
    dymu_ctx** ctxs;
    uint32_t n_ctx, n_goals;
    const uint32_t *goal_i, *goal_j;
    const double* start_xy;
    double tau;
    double* paths;
    uint32_t cap;
    uint32_t* path_len;
    int32_t* path_status;
    std::vector<int> rc;
    std::vector<float> ms;
};

struct BatchThread
{
    BatchShared* s;
    uint32_t k;
};

void* batch_worker(void* arg)
{
    BatchThread* t = (BatchThread*)arg;
    BatchShared& S = *t->s;
    const uint32_t k = t->k;
    dymu_ctx* ctx = S.ctxs[k];
    dymu_device_guard guard(ctx->device);
    // contiguous block of queries (sizes differ by at most one)
    const uint32_t base = S.n_goals / S.n_ctx, extra = S.n_goals % S.n_ctx;
    const uint32_t lo = k * base + (k < extra ? k : extra), cnt = base + (k < extra ? 1u : 0u);
    const uint32_t B = ctx->n_slots;
    std::vector<uint32_t> slots(B), gij(2 * (size_t)B);
    int rc = DYMU_OK;
    const double t0 = now_ms();
    for (uint32_t q0 = 0; q0 < cnt && rc == DYMU_OK; q0 += B)
    {
        const uint32_t m = (cnt - q0 < B) ? cnt - q0 : B;
        dymu_solve_stats st;
        rc = dymu_solve_total_cost(ctx, m, S.goal_i + lo + q0, S.goal_j + lo + q0, &st);
        if (rc != DYMU_OK || !S.start_xy || !S.paths) continue;
        for (uint32_t s = 0; s < m; ++s)
        {
            slots[s] = s;
            gij[2 * s] = S.goal_i[lo + q0 + s];
            gij[2 * s + 1] = S.goal_j[lo + q0 + s];
        }
        rc = dymu_extract_global_path_batch(ctx, m, slots.data(), S.start_xy + 2 * (size_t)(lo + q0), S.tau,
                                            gij.data(), S.paths + (size_t)(lo + q0) * S.cap * 5, S.cap,
                                            S.path_len + lo + q0, (int*)S.path_status + lo + q0);
    }
    if (rc == DYMU_OK) rc = dymu_synchronize(ctx);
    S.ms[k] = (float)(now_ms() - t0);
    S.rc[k] = rc;
    return nullptr;
}
}  // namespace

extern "C" {

int dymu_dd_solve(dymu_ctx** ctxs, uint32_t n, const uint32_t* cuts, uint32_t goal_i, uint32_t goal_j,
                  uint32_t phases_per_round, dymu_dd_stats* stats)
{
    if (!ctxs || n < 1 || !cuts) return DYMU_ERR_ARG;
    if (phases_per_round == 0) phases_per_round = 32;
    for (uint32_t k = 0; k < n; ++k)
    {
        if (!ctxs[k] || cuts[k + 1] <= cuts[k]) return DYMU_ERR_ARG;
        const uint32_t want = (cuts[k + 1] - cuts[k]) + (k > 0 ? 1u : 0u) + (k + 1 < n ? 1u : 0u);
        if (ctxs[k]->ny != want || ctxs[k]->nx != ctxs[0]->nx)
            DYMU_FAIL(ctxs[k], DYMU_ERR_ARG, "strip %u must have %u rows (own rows + ghost rows) and the common width", k,
                      want);
        if (!ctxs[k]->have_cost) DYMU_FAIL(ctxs[k], DYMU_ERR_STATE, "strip %u has no cost map", k);
        if (ctxs[k]->aniso_n)
            DYMU_FAIL(ctxs[k], DYMU_ERR_STATE, "strip %u: domain decomposition is isotropic only", k);
        if (ctxs[k]->clear_on)
            DYMU_FAIL(ctxs[k], DYMU_ERR_STATE, "strip %u: a strip cannot see obstacles across a cut (obstacle clearance)", k);
    }
    if (goal_i >= ctxs[0]->nx || goal_j < cuts[0] || goal_j >= cuts[n]) return DYMU_ERR_ARG;
    DdShared S;
    S.ctxs = ctxs; S.n = n; S.cuts = cuts; S.goal_i = goal_i; S.goal_j = goal_j; S.phases = phases_per_round;
    S.max_rounds = 1u << 20;
    S.inbox.assign(n, nullptr);
    S.sent.assign(n, nullptr);
    S.busy.assign(n, 0);
    S.rc.assign(n, DYMU_OK);
    S.kernel_ms.assign(n, 0.f);
    S.activations.assign(n, 0ull);
    S.updates.assign(n, 0ull);
    S.rounds = 0;
    S.any_failed = 0;
    int rc = DYMU_OK;
    for (uint32_t k = 0; k < n && rc == DYMU_OK; ++k)
    {
        dymu_device_guard guard(ctxs[k]->device);
        // direct stores into the neighbours' memory where the topology allows it (NVLink /
        // NVSwitch); otherwise the runtime stages the peer copies itself
        for (int d = -1; d <= 1; d += 2)
        {
            const long q = (long)k + d;
            if (q < 0 || q >= (long)n || ctxs[q]->device == ctxs[k]->device) continue;
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, ctxs[k]->device, ctxs[q]->device) == cudaSuccess && can)
            {
                cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[q]->device, 0);
                if (e != cudaSuccess) cudaGetLastError();  // already enabled: fine
            }
        }
        if (cudaMalloc((void**)&S.inbox[k], 2 * (size_t)ctxs[k]->nx * sizeof(double)) != cudaSuccess
            || cudaEventCreateWithFlags(&S.sent[k], cudaEventDisableTiming) != cudaSuccess)
        {
            snprintf(ctxs[k]->err, sizeof(ctxs[k]->err), "dymu_dd_solve: %s", cudaGetErrorString(cudaGetLastError()));
            rc = DYMU_ERR_CUDA;
        }
    }
    double t0 = now_ms(), t1 = t0;
    if (rc == DYMU_OK)
    {
        pthread_barrier_init(&S.bar, nullptr, n);
        std::vector<pthread_t> th(n);
        std::vector<DdThread> args(n);
        t0 = now_ms();
        for (uint32_t k = 0; k < n; ++k)
        {
            args[k].s = &S;
            args[k].k = k;
            pthread_create(&th[k], nullptr, dd_worker, &args[k]);
        }
        for (uint32_t k = 0; k < n; ++k) pthread_join(th[k], nullptr);
        t1 = now_ms();
        pthread_barrier_destroy(&S.bar);
        for (uint32_t k = 0; k < n; ++k)
            if (S.rc[k] != DYMU_OK && rc == DYMU_OK) rc = S.rc[k];
    }
    for (uint32_t k = 0; k < n; ++k)
    {
        dymu_device_guard guard(ctxs[k]->device);
        if (S.inbox[k]) cudaFree(S.inbox[k]);
        if (S.sent[k]) cudaEventDestroy(S.sent[k]);
    }
    if (stats)
    {
        memset(stats, 0, sizeof(*stats));
        stats->rounds = S.rounds;
        stats->converged = (rc == DYMU_OK) ? 1u : 0u;
        stats->wall_ms = (float)(t1 - t0);
        for (uint32_t k = 0; k < n; ++k)
        {
            if (S.kernel_ms[k] > stats->max_kernel_ms) stats->max_kernel_ms = S.kernel_ms[k];
            stats->sum_kernel_ms += S.kernel_ms[k];
            stats->tile_activations += S.activations[k];
            stats->cell_updates += S.updates[k];
        }
    }
    return rc;
}

int dymu_batch_solve(dymu_ctx** ctxs, uint32_t n_ctx, uint32_t n_goals, const uint32_t* goal_i,
                     const uint32_t* goal_j, const double* start_xy, double tau, double* paths, uint32_t cap,
                     uint32_t* path_len, int32_t* path_status, float* ms_per_ctx)
{
    if (!ctxs || n_ctx < 1 || !goal_i || !goal_j) return DYMU_ERR_ARG;
    if (paths && (!start_xy || !path_len || !path_status || cap == 0)) return DYMU_ERR_ARG;
    for (uint32_t k = 0; k < n_ctx; ++k)
        if (!ctxs[k]) return DYMU_ERR_ARG;
    if (n_goals == 0) return DYMU_OK;
    BatchShared S;
    S.ctxs = ctxs; S.n_ctx = n_ctx; S.n_goals = n_goals; S.goal_i = goal_i; S.goal_j = goal_j;
    S.start_xy = start_xy; S.tau = tau; S.paths = paths; S.cap = cap; S.path_len = path_len;
    S.path_status = path_status;
    S.rc.assign(n_ctx, DYMU_OK);
    S.ms.assign(n_ctx, 0.f);
    std::vector<pthread_t> th(n_ctx);
    std::vector<BatchThread> args(n_ctx);
    for (uint32_t k = 0; k < n_ctx; ++k)
    {
        args[k].s = &S;
        args[k].k = k;
        pthread_create(&th[k], nullptr, batch_worker, &args[k]);
    }
    int rc = DYMU_OK;
    for (uint32_t k = 0; k < n_ctx; ++k)
    {
        pthread_join(th[k], nullptr);
        if (S.rc[k] != DYMU_OK && rc == DYMU_OK) rc = S.rc[k];
        if (ms_per_ctx) ms_per_ctx[k] = S.ms[k];
    }
    return rc;
}

}  // extern "C"
