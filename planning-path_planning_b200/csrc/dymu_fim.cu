// dymu_fim.cu -- tiled Fast Iterative Method for the DyMu wave propagations.
//
// Replaces the reference's sequential Fast Marching loop (narrow band held in an
// unsorted std::vector with a linear argmin scan and vector::erase per pop,
// src/DyMu_GlobalPathPlanning.cpp:443-468, 551-568) by a fixed-point iteration of the
// very same node update (propagateGlobalNode, G.cpp:500-546):
//
//     Tx = min(T[i-1], T[i+1]);  Ty = min(T[j-1], T[j+1]);  C = ceff[j][i]
//     Tn = |Tx-Ty| < C && both finite ? (Tx+Ty+sqrt(2C^2-(Tx-Ty)^2))/2 : min(Tx,Ty)+C
//     T  = min(T, Tn)
//
// The FMM result is a fixed point of that update (a CLOSED node's value only depends on
// neighbours with smaller values), and the monotone iteration from T = +inf, T(goal) = 0
// converges to it from above, so both agree to rounding (DESIGN.md section 4).
//
// Execution model (one persistent cooperative launch per solve):
//   * the plane is cut into TILE x TILE tiles; a global work list holds the ACTIVE tiles;
//   * each CTA repeatedly takes a tile, stages T (+1-cell halo) and the cost term C in
//     shared memory, relaxes it there until nothing changes (or an iteration cap), writes
//     T back and, for every tile edge whose cells changed, appends the neighbouring tile
//     to the next list (deduplicated by an atomic flag word whose bits say WHICH halo of
//     the neighbour went stale);
//   * inside a tile, work is tracked per 8x8-cell block, one block per warp (two cells per
//     lane): a warp only re-evaluates its block if it is marked dirty (a cell of it or of the
//     facing edge of a neighbouring block changed in the previous sweep).  One warp-wide OR
//     (REDUX) of per-lane wake masks tells which blocks and tile edges a sweep touched; the
//     16-bit dirty masks rotate through three shared words, one __syncthreads per sweep.  A
//     wave crossing a tile therefore costs work proportional to the front length, not the
//     tile area;
//   * every wake-up carries the smallest changed value as a priority key; a phase only
//     relaxes the tiles whose key lies within a band above the smallest pending key, the
//     others are carried over untouched (far fewer sweeps with halos that are not final yet);
//   * phases are separated by a grid-wide barrier; three rotating lists let one be
//     reset while the next is filled;
//   * a solve can be stopped after a bounded number of phases and continued later
//     (dymu_solve_start / dymu_solve_advance): the lists stay consistent at phase boundaries.
// Host side: each caller starts the work lists itself -- dymu_internal_fim_clear and then k_seed
// (goals), k_seed_rows (tile rows) or k_seed_all (every tile), or, when continuing, the pending lists
// with rows merged in by k_seed_rows_add -- and dymu_internal_fim_run launches the kernel on them and
// decodes the statistics block (kStat* slots, dymu_ctx.cuh).
// Environment switch, read per call: DYMU_STREAM_PHASES (streamed solves cut after n / 2n phases
// instead of on the copy engine's word).  Build-time: -DDYMU_FIM_PROFILE (clock64 section profile,
// and the per-phase, per-CTA timeline that DYMU_FIM_CTA_TRACE names a file for).
// Direct delivery (dymu_set_total_cost_export): the kernel tracks an upper bound per tile and
// stores a tile into the caller's page-locked matrix once that bound is below every pending key
// (see Params::tmax); k_deliver_rest stores what is left.  A waiting CTA gives up after eight
// seconds at the grid barrier (barrier_spin) and the solve returns an error instead of hanging.
// The same kernel runs the local layer's risk dilation (propagateRisk,
// src/DyMu_LocalPathRepairing.cpp:550-576) in MODE 1, a max-propagation on risk, and a batch of
// independent maps (dymu_solve_maps) in MODE 3: MODE 0 with problem q reading its own cost-term
// plane at C + q * slot_stride.  MODE 4 is the anisotropic map batch: MODE 2 with the directional
// costs staged as C_q(x) * A_d(x), C_q read as in MODE 3 and A the four factor planes f(theta(x->m)).
#include <cooperative_groups.h>
#include <stdlib.h>

#include "dymu_ctx.cuh"

namespace
{
constexpr int TILE = kTile;  // (signed: the kernel's cell arithmetic is int)
static_assert(TILE == 32, "4 x 4 blocks of 8 x 8 cells");
constexpr int ROUNDS = 6;  // red-black rounds per block visit (an unchanged block stops early)
constexpr int WARPS = 16;  // one 8 x 8 block per warp
constexpr int THREADS = 32 * WARPS;
constexpr int BX = TILE / 8;       // 4 x 4 blocks of 8 x 8 cells, block w <-> warp w
constexpr int BY = TILE / 8;
// row pitch of the shared arrays in doubles.  A half-warp (what one 64-bit shared-memory
// transaction serves) touches four consecutive rows of a block, every other column of each
// (red-black ownership, see k_fim): with 36 doubles = 72 words per row the rows start 8
// banks apart and the four groups of alternate columns fall into disjoint banks
constexpr int PITCH = TILE + 4;
constexpr int CPT = TILE * TILE / THREADS;  // cells per thread in load/store = 2
constexpr int MIN_CTAS = 2;  // 1024 threads per SM: caps a thread at 64 registers
constexpr int SWEEP_CAP = 2 * TILE;  // sweeps per activation; the rest resumes next phase
constexpr size_t SMEM = sizeof(double) * ((TILE + 2) * PITCH + TILE * PITCH);
// MODE 2 / 4 stage the four directional costs of the tile instead of one cost term
constexpr size_t SMEM_ANISO = sizeof(double) * ((TILE + 2) * PITCH + 4 * TILE * PITCH);

// activation flag bits: which halo of the tile is stale / whole tile must be re-evaluated
constexpr uint32_t kHaloTop = 1u, kHaloBottom = 2u, kHaloLeft = 4u, kHaloRight = 8u, kFull = 16u,
                   kResume = 32u;  // kResume: continue from the dirty mask saved in dsave[tile]

struct Params
{
    double* T;
    size_t slot_stride;
    const double* C;
    uint32_t pitch, rows, ntx, nty, nprob;
    uint32_t* list0;
    uint32_t* list1;
    uint32_t* list2;
    uint32_t* flag0;
    uint32_t* flag1;
    uint32_t* flag2;
    unsigned long long* key0;   // per tile: smallest value among the changes it was woken for
    unsigned long long* key1;
    unsigned long long* key2;
    unsigned long long* gmin;   // [3] minimum key over each list
    uint32_t* dsave;            // per tile: dirty-block mask left over when the sweep cap hit
    unsigned long long* cta_trace;  // optional (profile build): per phase x CTA timeline
    uint32_t cta_trace_phases;
    uint32_t* ctrl;
    unsigned long long* stats;
    int max_outer;
    int outer0;                 // rotation of the three lists at entry (phase-bounded solves)
    double band;                // tiles with key > min key + band wait (inf = plain FIM)
    // direct delivery (MODE 0, one problem).  tmax[tile]: bit pattern of an upper bound of the tile's
    // values as of its last write-back, +inf while a passable cell is unreached, kExported once the
    // tile has been stored to xout.  A tile whose bound lies below the smallest pending key can no
    // longer change (the update is upwind: whatever a pending change produces is larger than it).
    unsigned long long* tmax;   // nullptr: not tracked
    double* xout;               // page-locked host matrix as the device sees it; nullptr: no delivery
    size_t xld;
    uint32_t xnx, xny;          // logical size (the plane is padded to whole tiles)
    int xminus1;                // +inf is delivered as -1 (getTotalCostMatrix, G.cpp:799-811)
    const uint32_t* stop_flag;  // leave after the phase in which *stop_flag >= stop_value (nullptr: never)
    uint32_t stop_value;
    // MODE 2: the directional costs a(x->m), four planes in the order i-1, i+1, j-1, j+1;
    // MODE 4: the factors f(theta(x->m)) in the same order, shared by all problems
    const double* A;
    size_t a_stride;            // doubles between two of those planes
};
constexpr unsigned long long kExported = 0xFFFFFFFFFFFFFFFFull;

__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p)
{
    return *reinterpret_cast<const volatile uint32_t*>(p);
}
__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long* p)
{
    return *reinterpret_cast<const volatile unsigned long long*>(p);
}
__device__ __forceinline__ void smem_or(uint32_t* p, uint32_t v)
{
    asm volatile("red.shared.or.b32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(p)), "r"(v) : "memory");
}
constexpr unsigned long long kNoKey = 0xFFFFFFFFFFFFFFFFull;
// non-negative doubles order like their bit patterns, so atomicMin on the bits is a min
__device__ __forceinline__ unsigned long long key_of(double v)
{
    return (unsigned long long)__double_as_longlong(v);
}

// Waits until *counter >= target.  A grid that lost a CTA (a defect, not a load condition) would
// spin here for ever and take the GPU with it: after about eight seconds of waiting the CTA gives
// up and says so in *abort_flag, which makes every other waiting CTA give up as well; the host
// reports the solve as failed.
// (not inlined: its loop state would otherwise take registers from the sweep)
__device__ __noinline__ bool barrier_spin(const uint32_t* counter, uint32_t target,
                                          unsigned long long* abort_flag)
{
    uint32_t polls = 0;
    unsigned long long t0 = 0;
    while (ld_volatile_u32(counter) < target)
    {
        if ((++polls & 0x3FFFu) == 0)
        {
            if (ld_volatile_u64(abort_flag)) return false;
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 8000000000ull)
            {
                *abort_flag = 1ull;
                __threadfence();
                return false;
            }
        }
    }
    return true;
}

// grid-wide barrier on a monotonically increasing arrival counter (all CTAs are
// co-resident: the kernel is launched with cudaLaunchCooperativeKernel).  `ok` is a word in
// shared memory; the return value (false: the grid is being abandoned) is the same for the whole CTA.
__device__ __forceinline__ bool grid_barrier(uint32_t* counter, uint32_t& phase, unsigned long long* abort_flag,
                                             uint32_t* ok)
{
    __syncthreads();
    if (threadIdx.x == 0)
    {
        __threadfence();
        uint32_t target = (phase + 1) * gridDim.x;
        atomicAdd(counter, 1u);
        *ok = barrier_spin(counter, target, abort_flag) ? 1u : 0u;
        __threadfence();
    }
    phase++;
    __syncthreads();
    return *ok != 0;
}

// the same barrier in two halves, so that a CTA can do work nobody waits for in between
__device__ __forceinline__ void grid_barrier_arrive(uint32_t* counter, uint32_t phase, uint32_t* order)
{
    __syncthreads();
    if (threadIdx.x == 0)
    {
        __threadfence();
        *order = atomicAdd(counter, 1u) - phase * gridDim.x;  // how many CTAs arrived before this one
    }
}
__device__ __forceinline__ bool grid_barrier_wait(uint32_t* counter, uint32_t& phase, unsigned long long* abort_flag,
                                                  uint32_t* ok)
{
    if (threadIdx.x == 0)
    {
        uint32_t target = (phase + 1) * gridDim.x;
        *ok = barrier_spin(counter, target, abort_flag) ? 1u : 0u;
        __threadfence();
    }
    phase++;
    __syncthreads();
    return *ok != 0;
}

template <int MODE> __device__ __forceinline__ double outside_value()
{
    return MODE == 1 ? 0.0 : DYMU_INF;  // missing neighbour: skipped (G.cpp:504-523) / risk 0 (L.cpp:555-558)
}

// min / max of two non-negative doubles through their bit patterns (identical to fmin/fmax
// for the values that occur here: finite >= 0 or +inf, never NaN) -- two integer
// instructions instead of a DSETP + select chain on the critical path
__device__ __forceinline__ double min_nn(double a, double b)
{
    long long x = __double_as_longlong(a), y = __double_as_longlong(b);
    return __longlong_as_double(x < y ? x : y);
}
__device__ __forceinline__ double max_nn(double a, double b)
{
    long long x = __double_as_longlong(a), y = __double_as_longlong(b);
    return __longlong_as_double(x > y ? x : y);
}

// One node update; returns true when the stored value improves.  Written branch-free so a
// warp stays converged and two blocks can be interleaved: the two-sided (sqrt) value is
// computed for every lane and selected afterwards.  The value it
// produces is bit-identical to propagateGlobalNode's (G.cpp:527-535):
//   * `Tx < inf && Ty < inf` is implied by |Tx-Ty| < C for finite C (inf-inf is NaN);
//   * C = +inf marks cells that are never targets (obstacles, padding): no update.
template <int MODE>
__device__ __forceinline__ bool relax(double tc, double tl, double tr, double tu, double td,
                                      double c, double cc2 /* 2 c^2 */, double& out)
{
    if (MODE != 1)  // MODE 0 / 3
    {
        // No guards around the square root: the argument 2c^2 - d^2 lies in [c^2, 2c^2] whenever
        // the two-sided value is selected; otherwise (one side +inf, both +inf -> d NaN, or a
        // non-target cell with c = +inf) the root is garbage or NaN, which is either not
        // selected or fails the final '<'.  dymu_sqrt_normal is branch-free, so junk arguments
        // cost nothing.
        const double Tx = min_nn(tl, tr), Ty = min_nn(td, tu);
        const double d = Tx - Ty;
        const bool two = fabs(d) < c;             // false for NaN d (both inf) and for d = +-inf
        const double t2 = (Tx + Ty + dymu_sqrt_normal(cc2 - (d * d))) * 0.5;
        const double t1 = min_nn(Tx, Ty) + c;
        const double Tn = two ? t2 : t1;
        out = Tn;
        return Tn < tc;  // c = +inf (obstacle, padding): Tn is +inf or NaN, never smaller
    }
    else
    {
        // propagateRisk, L.cpp:550-576; obstacle cells are never targets (c = +inf)
        const double Ry = max_nn(tu, td), Rx = max_nn(tl, tr);
        const double Sx = 1 - Rx, Sy = 1 - Ry;
        const double d = Sx - Sy;
        const bool target = c < DYMU_INF;
        const bool two = fabs(d) < c;
        double arg = (two && target) ? (2 * (c * c) - (d * d)) : 1.0;
        asm volatile("" : "+d"(arg));
        const double s2 = (Sx + Sy + dymu_sqrt_normal(arg)) / 2;
        const double s1 = fmin(Sx, Sy) + c;
        const double S = two ? s2 : s1;
        const double R = fmax(1 - S, 0.0);
        out = R;
        return target && (R > 0) && (R > tc);
    }
}

// MODE 2, the two-sided value of one neighbour pair: the root t of
//     ((t - Th) / ah)^2 + ((t - Tv) / av)^2 = 1
// when -ah < Th - Tv < av (exactly the condition t >= max(Th, Tv)), else +inf.  Expression order
// (restated by the test oracle; no contraction, correctly rounded sqrt and division):
//     d = Th - Tv; ah2 = ah*ah; av2 = av*av; s = ah2 + av2
//     t = ((av2*Th + ah2*Tv) + (ah*av)*sqrt(s - d*d)) / s
// With ah = av = C this is the isotropic update of G.cpp:527-535 up to rounding.  An infinite
// ah or av (impassable cell, neighbour outside the grid) or an infinite Th / Tv never gives a
// valid pair; the square root of a junk argument is not selected (dymu_sqrt_normal is branch-free).
__device__ __forceinline__ double aniso_pair(double Th, double ah, double Tv, double av)
{
    const double d = Th - Tv;
    const double ah2 = ah * ah, av2 = av * av;
    const double s = ah2 + av2;
    const bool valid = (d > -ah) && (d < av) && (s < DYMU_INF);
    const double t = ((av2 * Th + ah2 * Tv) + (ah * av) * dymu_sqrt_normal(s - d * d)) / s;
    return valid ? t : DYMU_INF;
}

// MODE 2 node update: the smallest of the four one-sided values T[m] + a(x->m) and the four
// two-sided pair values, against the stored value as in MODE 0.  `ac` points at the cell's
// directional cost toward i-1 in shared memory; the other three follow at `ps` doubles each.
// Every candidate is >= 0 or +inf (never NaN), so the minima are taken on the bit patterns.
__device__ __forceinline__ bool relax_aniso(double tc, double txm, double txp, double tym, double typ,
                                            const double* ac, int ps, double& out)
{
    const double axm = ac[0], axp = ac[ps], aym = ac[2 * ps], ayp = ac[3 * ps];
    double Tn = min_nn(min_nn(txm + axm, txp + axp), min_nn(tym + aym, typ + ayp));
    Tn = min_nn(Tn, min_nn(aniso_pair(txm, axm, tym, aym), aniso_pair(txm, axm, typ, ayp)));
    Tn = min_nn(Tn, min_nn(aniso_pair(txp, axp, tym, aym), aniso_pair(txp, axp, typ, ayp)));
    out = Tn;
    return Tn < tc;  // an impassable cell has every candidate +inf: never smaller
}

template <int MODE>
__global__ void __launch_bounds__(THREADS, MIN_CTAS) k_fim(Params p)
{
    constexpr int P = PITCH;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* Ts = reinterpret_cast<double*>(smem_raw);            // (TILE+2) x P, 1-cell halo
    double* Cs = Ts + (TILE + 2) * P;                            // TILE x P
    // dirty 8x8 blocks for the next sweep: every warp posts what its block visit woke up into its own
    // word (plain store, two sets alternating by sweep parity); after the barrier each warp ORs the
    // sixteen words with one warp reduction -- no shared-memory atomics in the sweep
    __shared__ uint32_t s_post[2][WARPS];
    __shared__ uint32_t s_m0;      // dirty set an activation starts with
    __shared__ uint32_t edge_mask;  // tile edges with a changed cell: 1 top, 2 bottom, 4 left, 8 right
    __shared__ uint32_t s_tile;
    __shared__ unsigned long long s_emin[5];  // min changed value per edge [0..3], overall [4]
    __shared__ uint32_t s_tmax;                // high word (rounded up) of the largest passable value
    __shared__ uint32_t s_xtile;               // the tile this CTA delivers in the current phase
    __shared__ uint32_t s_xorder;              // its order of arrival at the barrier
    __shared__ uint32_t s_bar_ok;              // grid barrier: 0 when the grid is being abandoned

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t tiles_per_prob = p.ntx * p.nty;
    // ---- per-thread constants of the sweep.  Warp w owns the 8x8 block w
    // (bx = w & 3, by = w >> 2); lane (lx, ly) owns the two cells (lx, 2 ly) and (lx, 2 ly + 1) of
    // it, one of each colour of the checkerboard (x + y even = red).  A block visit relaxes the
    // red cells of the block first and the black ones after a __syncwarp, so the black cells see
    // this very visit's red values: information moves two cells per sweep instead of one
    // (red-black Gauss-Seidel inside the block, Jacobi between the blocks), which halves the
    // sweeps a wave needs to cross a tile at the same instruction count per sweep.
    // wake.x / wake.y: what a change of the lane's first (red) / second (black) cell has to wake
    // up -- the own block, the neighbour block across a block edge (bits 0..15) and the tile
    // edge the cell sits on (bits 16..19: top, bottom, left, right).
    // The masks live in shared memory: kept in registers the compiler re-derives them from the
    // thread index in every sweep (64-register cap), which costs more issue slots than one load.
    constexpr int c_off = (TILE + 1) * P - 1;  // from a cell of Ts to the same cell of Cs
    __shared__ uint2 s_wake[THREADS];
    double* cell1;          // the lane's red cell
    int to_second;          // offset (doubles) from the red to the black cell: +P or -P
    uint32_t my_bit;
    {
        const int lx = lane & 7, ly = lane >> 3;
        const bool upper_is_red = (lx & 1) == 0;  // rows 2 ly (upper) and 2 ly + 1 (lower)
        to_second = upper_is_red ? P : -P;
        asm volatile("" : "+r"(to_second));
        const int bx = warp & 3, by = warp >> 2;
        // opaque offset: otherwise it is re-derived from the thread index in every sweep
        int off = (by * 8 + 2 * ly + (upper_is_red ? 0 : 1) + 1) * P + bx * 8 + lx + 1;
        asm volatile("" : "+r"(off));
        cell1 = Ts + off;
        my_bit = 1u << warp;
        const uint32_t bitL = bx > 0 ? my_bit >> 1 : 0x40000u, bitR = bx < BX - 1 ? my_bit << 1 : 0x80000u;
        const uint32_t bitU = by > 0 ? my_bit >> 4 : 0x10000u, bitD = by < BY - 1 ? my_bit << 4 : 0x20000u;
        const uint32_t side = (lx == 0 ? bitL : 0u) | (lx == 7 ? bitR : 0u);
        const uint32_t w_upper = my_bit | side | (ly == 0 ? bitU : 0u);
        const uint32_t w_lower = my_bit | side | (ly == 3 ? bitD : 0u);
        s_wake[tid] = upper_is_red ? make_uint2(w_upper, w_lower) : make_uint2(w_lower, w_upper);
    }
    auto sel3 = [](uint32_t* a, uint32_t* b, uint32_t* c, int k) { return k == 0 ? a : (k == 1 ? b : c); };
    auto sel3k = [](unsigned long long* a, unsigned long long* b, unsigned long long* c, int k) {
        return k == 0 ? a : (k == 1 ? b : c);
    };
    // direct delivery: one tile of the plane to the caller's matrix
    auto deliver_tile = [&](uint32_t t) {
        const uint32_t ty = t / p.ntx, tx = t - ty * p.ntx;
#pragma unroll
        for (int k = 0; k < CPT; ++k)
        {
            const int e = tid + k * THREADS;
            const uint32_t gy = ty * TILE + e / TILE, gx = tx * TILE + e % TILE;
            if (gx < p.xnx && gy < p.xny)
            {
                double v = __ldcg(&p.T[(size_t)gy * p.pitch + gx]);
                if (p.xminus1 && v == DYMU_INF) v = -1.0;
                p.xout[(size_t)gy * p.xld + gx] = v;
            }
        }
    };
    uint32_t phase = 0;
    unsigned long long n_tiles = 0, n_visits = 0, n_deferred = 0, n_inner = 0;
    uint32_t n_written = 0;  // cells this thread stored back to the plane
#ifdef DYMU_FIM_PROFILE
    long long pc_fetch = 0, pc_load = 0, pc_sweep = 0, pc_store = 0, pc_barrier = 0, pc_t = clock64();
#define PC_MARK(acc) { long long now__ = clock64(); acc += now__ - pc_t; pc_t = now__; }
    unsigned long long tl_fetch = 0, tl_load = 0, tl_sweep = 0, tl_store = 0, tl_tiles = 0, tl_start = 0;
#define GT(var) { unsigned long long g__; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g__)); var = g__; }
#else
#define PC_MARK(acc)
#endif
    int outer = p.outer0;
    bool converged = false;

    for (; outer < p.outer0 + p.max_outer; ++outer)
    {
        const int cur = outer % 3, nxt = (outer + 1) % 3, old = (outer + 2) % 3;
        const uint32_t n_active = ld_volatile_u32(&p.ctrl[kCtrlCount + cur]);
        if (n_active == 0)
        {
            converged = true;
            break;
        }
        if (p.stop_flag)
        {
            // Asked to hand back?  ctrl[kCtrlStopAt] holds the iteration BEFORE which every CTA leaves:
            // CTA 0 writes it ahead of its arrival at a barrier, and it may already be running one phase
            // ahead of a CTA that is slow to leave that barrier -- a plain flag would make the slow
            // one leave a phase early and the others wait for it forever.
            const uint32_t stop_at = ld_volatile_u32(&p.ctrl[kCtrlStopAt]);
            if (stop_at != 0 && stop_at <= (uint32_t)outer + 1u) break;
        }
#ifdef DYMU_FIM_PROFILE
        if (tid == 0) { GT(tl_start) tl_fetch = tl_load = tl_sweep = tl_store = tl_start; tl_tiles = 0; }
#endif
        uint32_t* list_cur = sel3(p.list0, p.list1, p.list2, cur);
        uint32_t* list_nxt = sel3(p.list0, p.list1, p.list2, nxt);
        uint32_t* flag_cur = sel3(p.flag0, p.flag1, p.flag2, cur);
        uint32_t* flag_nxt = sel3(p.flag0, p.flag1, p.flag2, nxt);
        unsigned long long* key_cur = sel3k(p.key0, p.key1, p.key2, cur);
        unsigned long long* key_nxt = sel3k(p.key0, p.key1, p.key2, nxt);
        // priority band: only tiles whose pending information is within `band` of the
        // smallest pending value anywhere are relaxed in this phase; the others are carried
        // to the next list untouched.  This keeps tiles from being swept with halo values
        // that are still far from final (the source of most re-activations in plain FIM).
        unsigned long long limit = kNoKey;
        {
            const unsigned long long gm = ld_volatile_u64(&p.gmin[cur]);
            const double lim = __longlong_as_double((long long)gm) + p.band;
            if (gm != kNoKey && lim < DYMU_INF) limit = key_of(lim);
        }

        bool first_fetch = true;
        for (;;)
        {
            __syncthreads();
            if (tid == 0)
            {
                uint32_t t = 0xffffffffu;
                for (;;)
                {
                    // the first gridDim.x entries of a phase are pre-assigned, one per CTA; the
                    // shared cursor only hands out the rest
                    uint32_t idx;
                    if (first_fetch)
                    {
                        idx = blockIdx.x;
                        first_fetch = false;
                    }
                    else
                    {
                        // no shared cursor to ask when every entry was pre-assigned
                        if (n_active <= gridDim.x) break;
                        idx = gridDim.x + atomicAdd(&p.ctrl[kCtrlCursor + cur], 1u);
                    }
                    if (idx >= n_active) break;
                    const uint32_t cand = ld_volatile_u32(&list_cur[idx]);
                    const unsigned long long k = ld_volatile_u64(&key_cur[cand]);
                    if (k <= limit)
                    {
                        t = cand;
                        break;
                    }
                    // defer: move flag bits and key to the next list
                    const uint32_t bits = ld_volatile_u32(&flag_cur[cand]);
                    flag_cur[cand] = 0;
                    key_cur[cand] = kNoKey;
                    atomicMin(&key_nxt[cand], k);
                    atomicMin(&p.gmin[nxt], k);
                    if (atomicOr(&flag_nxt[cand], bits) == 0)
                        list_nxt[atomicAdd(&p.ctrl[kCtrlCount + nxt], 1u)] = cand;
                    n_deferred++;
                }
                s_tile = t;
            }
            __syncthreads();
            PC_MARK(pc_fetch)
            const uint32_t tile_id = s_tile;
#ifdef DYMU_FIM_PROFILE
            if (tid == 0 && tile_id != 0xffffffffu && tl_tiles == 0) GT(tl_fetch)
#endif
            if (tile_id == 0xffffffffu) break;
            const uint32_t prob = tile_id / tiles_per_prob;
            const uint32_t trem = tile_id - prob * tiles_per_prob;
            const uint32_t ty = trem / p.ntx, tx = trem - ty * p.ntx;
            const uint32_t why = ld_volatile_u32(&flag_cur[tile_id]);
            double* Tg = p.T + (size_t)prob * p.slot_stride + (size_t)ty * TILE * p.pitch
                         + (size_t)tx * TILE;
            const double* Cg = p.C + (MODE == 3 || MODE == 4 ? (size_t)prob * p.slot_stride : 0)
                               + (size_t)ty * TILE * p.pitch + (size_t)tx * TILE;

            // ---- stage the tile: T interior + halo (L2-coherent loads: other CTAs write
            // T during this phase), C through the read-only path
            // All global loads of a thread are issued before the first one is consumed, so that
            // staging costs one memory round trip (the halo used to be a second one).
            static_assert(4 * TILE <= THREADS, "one halo cell per thread");
            double hv = outside_value<MODE>();
            int hslot = -1;
            if (tid < 4 * TILE)
            {
                const int side = tid / TILE, q = tid % TILE;
                const double* src = nullptr;
                if (side == 0)
                {
                    if (ty > 0) src = &Tg[-(ptrdiff_t)p.pitch + q];
                    hslot = q + 1;
                }
                else if (side == 1)
                {
                    if (ty + 1 < p.nty) src = &Tg[(size_t)TILE * p.pitch + q];
                    hslot = (TILE + 1) * P + q + 1;
                }
                else if (side == 2)
                {
                    if (tx > 0) src = &Tg[(size_t)q * p.pitch - 1];
                    hslot = (q + 1) * P;
                }
                else
                {
                    if (tx + 1 < p.ntx) src = &Tg[(size_t)q * p.pitch + TILE];
                    hslot = (q + 1) * P + TILE + 1;
                }
                if (src) hv = __ldcg(src);
            }
            double told[CPT];
#pragma unroll
            for (int k = 0; k < CPT; ++k)
            {
                int e = tid + k * THREADS;
                int y = e / TILE, x = e % TILE;
                double v = __ldcg(&Tg[(size_t)y * p.pitch + x]);
                told[k] = v;
                Ts[(y + 1) * P + x + 1] = v;
                if constexpr (MODE == 2)
                {
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        Cs[q * TILE * P + y * P + x] =
                            __ldg(&p.A[q * p.a_stride + (size_t)(ty * TILE + y) * p.pitch + tx * TILE + x]);
                }
                else if constexpr (MODE == 4)
                {
                    // k_dircost's a(x->m) = C_eff(x) * f, bit for bit: +inf for an impassable cell (C_q
                    // = +inf) and toward an outside neighbour (f = +inf), overflow included
                    const double c = __ldg(&Cg[(size_t)y * p.pitch + x]);
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        Cs[q * TILE * P + y * P + x] =
                            c * __ldg(&p.A[q * p.a_stride + (size_t)(ty * TILE + y) * p.pitch + tx * TILE + x]);
                }
                else
                    Cs[y * P + x] = __ldg(&Cg[(size_t)y * p.pitch + x]);
            }
            if (hslot >= 0) Ts[hslot] = hv;
            // initial dirty set: the blocks along the stale halos (+ what an interrupted
            // sweep left over), or everything for a seeded tile
            if (tid == 0)
            {
                uint32_t m0 = 0;
                if (why & kResume) m0 |= p.dsave[tile_id];
                if (why & kFull) m0 = 0xffffu;
                if (why & kHaloTop) m0 |= 0x000Fu;                           // by == 0
                if (why & kHaloBottom) m0 |= 0xF000u;                        // by == BY-1
                if (why & kHaloLeft) m0 |= 0x1111u;                          // bx == 0
                if (why & kHaloRight) m0 |= 0x8888u;                         // bx == BX-1
                s_m0 = m0;
                flag_cur[tile_id] = 0;  // consumed; writers use flag_nxt / key_nxt this phase
                key_cur[tile_id] = kNoKey;
            }
            if (tid == 0)
            {
                edge_mask = 0;
                s_tmax = 0;
            }
            if (tid < 5) s_emin[tid] = kNoKey;
            __syncthreads();
            PC_MARK(pc_load)
#ifdef DYMU_FIM_PROFILE
            if (tid == 0 && tl_tiles == 0) GT(tl_load)
#endif

            // ---- relax in shared memory.  Warp w owns the 8x8 block w (bx = w & 3, by = w >> 2);
            // lane (lx, ly) owns one red and one black cell of it (see above).  A sweep is
            // therefore one visit per warp, whatever the number of dirty blocks.
            int it = 0;
            uint32_t visits = 0;
            uint32_t m = s_m0;
            uint32_t edges_acc = 0;  // warp-uniform: tile edges this warp's block changed (bits 0..3)
            const double cA = cell1[c_off], cB = cell1[to_second + c_off];
            const double qA = 2 * (cA * cA), qB = 2 * (cB * cB);
            // one sweep: relax the warp's block if m lists it dirty; returns the next dirty set
            auto sweep = [&](uint32_t* post) -> uint32_t {
                uint32_t contrib = 0;
                if (m & my_bit)
                {
                    double* a = cell1;
                    double* b = a + to_second;
                    // requested with the cell values and pinned here: left to the compiler the
                    // load sinks below the update and its latency lands on the chain
                    uint2 wake = s_wake[tid];
                    asm volatile("" : "+r"(wake.x), "+r"(wake.y));
                    uint32_t woke = 0;
#pragma unroll
                    for (int round = 0; round < ROUNDS; ++round)
                    {
                        // red cells of the block ...
                        double tA = a[0];
                        const double lA = a[-1], rA = a[1], uA = a[-P], dA = a[P];
                        asm volatile("" : "+d"(tA));
                        double nA, nB;
                        bool chA;
                        if constexpr (MODE == 2 || MODE == 4)
                            chA = relax_aniso(tA, lA, rA, uA, dA, a + c_off, TILE * P, nA);
                        else
                            chA = relax<MODE>(tA, lA, rA, uA, dA, cA, qA, nA);
                        if (chA) a[0] = nA;
                        __syncwarp();
                        // ... then the black ones, on the red values just stored
                        const double tB = b[0];
                        const double lB = b[-1], rB = b[1], uB = b[-P], dB = b[P];
                        bool chB;
                        if constexpr (MODE == 2 || MODE == 4)
                            chB = relax_aniso(tB, lB, rB, uB, dB, b + c_off, TILE * P, nB);
                        else
                            chB = relax<MODE>(tB, lB, rB, uB, dB, cB, qB, nB);
                        if (chB) b[0] = nB;
                        woke |= (chA ? wake.x : 0u) | (chB ? wake.y : 0u);
                        visits += 2;
                        if (round + 1 < ROUNDS)
                        {
                            // another round only pays while the block is still changing
                            if (!__any_sync(0xffffffffu, chA || chB)) break;
                        }
                    }
                    // one warp reduction tells which blocks (bits 0..15) and which tile edges
                    // (bits 16..19) saw a change
                    contrib = __reduce_or_sync(0xffffffffu, woke);
                }
                edges_acc |= contrib >> 16;
                if (lane == 0) post[warp] = contrib & 0xffffu;
                __syncthreads();
                ++it;
                return __reduce_or_sync(0xffffffffu, post[lane & (WARPS - 1)]);
            };
            for (;;)
            {
                if (m == 0 || it >= SWEEP_CAP) break;
                m = sweep(s_post[0]);
                if (m == 0 || it >= SWEEP_CAP) break;
                m = sweep(s_post[1]);
            }
            if (edges_acc && lane == 0) smem_or(&edge_mask, edges_acc);
            n_visits += visits;
            const int more = (m != 0);
            if (more && tid == 0) p.dsave[tile_id] = m;
            PC_MARK(pc_sweep)
#ifdef DYMU_FIM_PROFILE
            if (tid == 0 && tl_tiles == 0) GT(tl_sweep)
#endif

            // ---- write back changed cells and wake the neighbours whose halo went stale
            uint32_t vmax = 0;  // direct delivery: high word, rounded up, of the largest passable value
            {
                // smallest new value per tile edge = the priority the neighbour gets; [4]: smallest
                // new value anywhere, the tile's own priority when it has to be continued
                unsigned long long kmin[5] = {kNoKey, kNoKey, kNoKey, kNoKey, kNoKey};
                bool any = false;
#pragma unroll
                for (int k = 0; k < CPT; ++k)
                {
                    int e = tid + k * THREADS;
                    int y = e / TILE, x = e % TILE;
                    double v = Ts[(y + 1) * P + x + 1];
                    if (MODE != 1 && p.tmax && Cs[y * P + x] < DYMU_INF)
                        vmax = max(vmax, (uint32_t)(key_of(v) >> 32) + 1u);
                    if (v != told[k])
                    {
                        n_written++;
                        __stcg(&Tg[(size_t)y * p.pitch + x], v);
                        if (MODE != 1)
                        {
                            // A neighbouring tile only has to look again if this cell dropped below
                            // the cell facing it across the edge: the update is upwind, a cell is
                            // never improved through a neighbour that is not smaller, and the halo
                            // value is an upper bound of what the facing cell holds by now.  This
                            // drops the wake-ups a tile would send to the tiles it was fed from.
                            const unsigned long long kb = key_of(v);
                            any = true;
                            if (y == 0 && v < Ts[x + 1]) kmin[0] = min(kmin[0], kb);
                            if (y == TILE - 1 && v < Ts[(TILE + 1) * P + x + 1]) kmin[1] = min(kmin[1], kb);
                            if (x == 0 && v < Ts[(y + 1) * P]) kmin[2] = min(kmin[2], kb);
                            if (x == TILE - 1 && v < Ts[(y + 1) * P + TILE + 1]) kmin[3] = min(kmin[3], kb);
                            if (more) kmin[4] = min(kmin[4], kb);
                        }
                    }
                }
                if (MODE != 1 && __any_sync(0xffffffffu, any))
                {
                    // one shared-memory atomic per warp and edge instead of one per cell (64-bit
                    // shared-memory minima are compare-and-swap loops)
#pragma unroll
                    for (int q = 0; q < 5; ++q)
                    {
                        const uint32_t hi = (uint32_t)(kmin[q] >> 32), lo = (uint32_t)kmin[q];
                        const uint32_t mhi = __reduce_min_sync(0xffffffffu, hi);
                        const uint32_t mlo = __reduce_min_sync(0xffffffffu, hi == mhi ? lo : 0xffffffffu);
                        const unsigned long long r = ((unsigned long long)mhi << 32) | mlo;
                        if (lane == 0 && r != kNoKey) atomicMin(&s_emin[q], r);
                    }
                }
            }
            if (MODE != 1 && p.tmax)
            {
                vmax = __reduce_max_sync(0xffffffffu, vmax);
                if (lane == 0 && vmax) atomicMax(&s_tmax, vmax);
            }
            // No fence here: the values and the wake-ups are consumed after the grid barrier,
            // whose arrival (bar.sync, then thread 0's cumulative fence) orders them; tiles that
            // read this one's cells during the same phase may see old or new values, both are
            // valid upper bounds.
            __syncthreads();
            if (tid < 5)
            {
                uint32_t target = 0xffffffffu, bit = 0;
                uint32_t em = edge_mask;
                if (MODE != 1)  // only the edges across which a value can actually travel
                    em = (s_emin[0] != kNoKey ? 1u : 0u) | (s_emin[1] != kNoKey ? 2u : 0u)
                         | (s_emin[2] != kNoKey ? 4u : 0u) | (s_emin[3] != kNoKey ? 8u : 0u);
                if (tid == 0 && (em & 1u) && ty > 0) { target = tile_id - p.ntx; bit = kHaloBottom; }
                if (tid == 1 && (em & 2u) && ty + 1 < p.nty) { target = tile_id + p.ntx; bit = kHaloTop; }
                if (tid == 2 && (em & 4u) && tx > 0) { target = tile_id - 1; bit = kHaloRight; }
                if (tid == 3 && (em & 8u) && tx + 1 < p.ntx) { target = tile_id + 1; bit = kHaloLeft; }
                if (tid == 4 && more) { target = tile_id; bit = kResume; }  // cap hit: not converged
                if (MODE != 1 && tid == 4 && p.tmax) p.tmax[tile_id] = (unsigned long long)s_tmax << 32;
                if (target != 0xffffffffu)
                {
                    unsigned long long kb = (MODE != 1) ? s_emin[tid] : 0ull;
                    if (kb == kNoKey) kb = 0ull;  // (cannot happen: a flagged edge has a changed cell)
                    atomicMin(&key_nxt[target], kb);
                    atomicMin(&p.gmin[nxt], kb);
                    if (atomicOr(&flag_nxt[target], bit) == 0)
                    {
                        uint32_t pos = atomicAdd(&p.ctrl[kCtrlCount + nxt], 1u);
                        list_nxt[pos] = target;
                    }
                }
            }
            n_tiles++;
            n_inner += (unsigned long long)it;
            PC_MARK(pc_store)
#ifdef DYMU_FIM_PROFILE
            if (tid == 0) { GT(tl_store) tl_tiles++; }
#endif
        }
        PC_MARK(pc_fetch)
#ifdef DYMU_FIM_PROFILE
        if (tid == 0 && p.cta_trace && (uint32_t)outer < p.cta_trace_phases)
        {
            unsigned long long tl_arrive; GT(tl_arrive)
            unsigned long long* o = p.cta_trace + ((size_t)outer * gridDim.x + blockIdx.x) * 8;
            o[0] = tl_start; o[1] = tl_fetch; o[2] = tl_load; o[3] = tl_sweep; o[4] = tl_store;
            o[5] = tl_arrive; o[6] = tl_tiles; o[7] = n_active;
        }
#endif
        if (blockIdx.x == 0 && tid == 0)
        {
            if (p.stop_flag && ld_volatile_u32(&p.ctrl[kCtrlStopAt]) == 0 && ld_volatile_u32(p.stop_flag) >= p.stop_value)
                p.ctrl[kCtrlStopAt] = (uint32_t)outer + 2u;  // = (next iteration) + 1, never 0
            p.ctrl[kCtrlCount + old] = 0;   // count of the list that becomes "next" after this barrier
            p.ctrl[kCtrlCursor + old] = 0;  // and its cursor
            p.gmin[old] = kNoKey;
        }
        if (MODE != 1 && p.xout)
        {
            // Between arriving at the barrier and leaving it, the CTAs that arrive in the first half
            // -- they would only wait -- look through the tile bounds (a share of the array each,
            // by order of arrival) and deliver one of the tiles the front has left behind.  The CTAs
            // the others are waiting for skip this, so a phase is not made longer.
            // One tile per CTA and phase keeps the delivery inside the time an early CTA would wait at
            // the barrier anyway (4096^2: solve 7.82 ms without, 7.90 ms with; 8.28 ms at 64 per phase);
            // the half of the grid that delivers still moves 148 tiles per phase, twice what finishes.
            // the smallest key that was pending when this phase began: every value below it is final.
            // Read BEFORE arriving -- nothing writes gmin[cur] during its own phase, but once this CTA
            // has arrived the others may run ahead and recycle that slot for the phase after next.
            const unsigned long long gm = ld_volatile_u64(&p.gmin[cur]);
            grid_barrier_arrive(&p.ctrl[kCtrlBarrier], phase, &s_xorder);
            if (tid == 0) s_xtile = 0xffffffffu;
            __syncthreads();
            const uint32_t order = s_xorder, sharers = max(gridDim.x / 2u, 1u);
            if (order < sharers)
            {
                const uint32_t per = (tiles_per_prob + sharers - 1) / sharers;
                const uint32_t t_end = min((order + 1) * per, tiles_per_prob);
                // the first final tile found is claimed; the others are found again next phase
                for (uint32_t t = order * per + tid; t < t_end; t += THREADS)
                    if (ld_volatile_u64(&p.tmax[t]) < gm && atomicCAS(&s_xtile, 0xffffffffu, t) == 0xffffffffu)
                        p.tmax[t] = kExported;
                __syncthreads();
                const uint32_t xt = s_xtile;
                if (xt != 0xffffffffu)
                {
                    deliver_tile(xt);
                    if (tid == 0) atomicAdd(&p.stats[kStatDelivered], 1ull);
                }
            }
            if (!grid_barrier_wait(&p.ctrl[kCtrlBarrier], phase, &p.stats[kStatAbort], &s_bar_ok)) break;
        }
        else if (!grid_barrier(&p.ctrl[kCtrlBarrier], phase, &p.stats[kStatAbort], &s_bar_ok))
            break;
        PC_MARK(pc_barrier)
    }
#ifdef DYMU_FIM_PROFILE
    if (tid == 0)
    {
        atomicAdd(&p.stats[kStatCycFetch], (unsigned long long)pc_fetch);
        atomicAdd(&p.stats[kStatCycLoad], (unsigned long long)pc_load);
        atomicAdd(&p.stats[kStatCycSweep], (unsigned long long)pc_sweep);
        atomicAdd(&p.stats[kStatCycStore], (unsigned long long)pc_store);
        atomicAdd(&p.stats[kStatCycBarrier], (unsigned long long)pc_barrier);
    }
#endif

    // ---- statistics
    if (lane == 0 && n_visits) atomicAdd(&p.stats[kStatVisits], n_visits);
    {
        const uint32_t w = __reduce_add_sync(0xffffffffu, n_written);
        if (lane == 0 && w) atomicAdd(&p.stats[kStatWritten], (unsigned long long)w);
    }
    if (tid == 0)
    {
        if (n_tiles) atomicAdd(&p.stats[kStatTiles], n_tiles);
        if (n_deferred) atomicAdd(&p.stats[kStatDeferred], n_deferred);
        if (n_inner) atomicAdd(&p.stats[kStatSweeps], n_inner);
        if (blockIdx.x == 0)
        {
            p.stats[kStatPhases] = (unsigned long long)(outer - p.outer0);
            p.stats[kStatConverged] = converged ? 1ull : 0ull;
        }
    }
}


// Direct delivery, the rest: what the solve kernel did not get to store into the caller's matrix --
// the tiles the front reached last and the ones it never reached.  Runs on the copy stream right
// behind a converged solve, next to whatever the caller does then (path extraction).
__global__ void __launch_bounds__(512) k_deliver_rest(const double* T, uint32_t pitch, uint32_t ntx, uint32_t nty,
                                                      unsigned long long* tmax, double* xout, size_t xld,
                                                      uint32_t xnx, uint32_t xny, int xminus1,
                                                      unsigned long long* stats)
{
    if (ld_volatile_u64(&stats[kStatConverged]) == 0) return;  // not converged: the plane is not final
    const uint32_t total = ntx * nty;
    for (uint32_t t = blockIdx.x; t < total; t += gridDim.x)
    {
        if (ld_volatile_u64(&tmax[t]) == kExported) continue;
        const uint32_t ty = t / ntx, tx = t - ty * ntx;
        for (uint32_t e = threadIdx.x; e < TILE * TILE; e += blockDim.x)
        {
            const uint32_t gy = ty * TILE + e / TILE, gx = tx * TILE + e % TILE;
            if (gx < xnx && gy < xny)
            {
                double v = __ldcg(&T[(size_t)gy * pitch + gx]);
                if (xminus1 && v == DYMU_INF) v = -1.0;
                xout[(size_t)gy * xld + gx] = v;
            }
        }
    }
}

// One thread seeds all goals (there are at most a few hundred).  A goal on an obstacle cell is not
// seeded and counted in stats[kStatGoalObstacle]: "The goal is not valid", G.cpp:370-374 / 447-451.
__global__ void k_seed(double* T, size_t slot_stride, uint32_t pitch, uint32_t ntx, uint32_t nty,
                       int tile, const uint32_t* goal_ij, uint32_t n, const uint8_t* obst, uint32_t* list0,
                       uint32_t* flag0, unsigned long long* key0, unsigned long long* gmin,
                       uint32_t* ctrl, unsigned long long* stats)
{
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    uint32_t n_seeded = 0;
    for (uint32_t q = 0; q < n; ++q)
    {
        uint32_t gi = goal_ij[2 * q], gj = goal_ij[2 * q + 1];
        if (obst && obst[(size_t)gj * pitch + gi])
        {
            stats[kStatGoalObstacle]++;
            continue;
        }
        T[(size_t)q * slot_stride + (size_t)gj * pitch + gi] = 0.0;  // resetGlobalNarrowBand, G.cpp:490-496
        uint32_t tile_id = q * ntx * nty + (gj / tile) * ntx + gi / tile;
        flag0[tile_id] = kFull;
        key0[tile_id] = 0ull;
        list0[n_seeded++] = tile_id;
    }
    ctrl[kCtrlCount] = n_seeded;
    if (n_seeded) gmin[0] = 0ull;
}

// k_seed for a map batch: goal q is tested against its own cost-term plane (C_eff = +inf: obstacle)
__global__ void k_seed_maps(double* T, size_t slot_stride, uint32_t pitch, uint32_t ntx, uint32_t nty,
                            const uint32_t* goal_ij, uint32_t n, const double* ceff, uint32_t* list0,
                            uint32_t* flag0, unsigned long long* key0, unsigned long long* gmin,
                            uint32_t* ctrl, unsigned long long* stats)
{
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    uint32_t n_seeded = 0;
    for (uint32_t q = 0; q < n; ++q)
    {
        const size_t cell = (size_t)goal_ij[2 * q + 1] * pitch + goal_ij[2 * q];
        if (!(ceff[(size_t)q * slot_stride + cell] < DYMU_INF))
        {
            stats[kStatGoalObstacle]++;
            continue;
        }
        T[(size_t)q * slot_stride + cell] = 0.0;
        const uint32_t tile_id = q * ntx * nty + (goal_ij[2 * q + 1] / TILE) * ntx + goal_ij[2 * q] / TILE;
        flag0[tile_id] = kFull;
        key0[tile_id] = 0ull;
        list0[n_seeded++] = tile_id;
    }
    ctrl[kCtrlCount] = n_seeded;
    if (n_seeded) gmin[0] = 0ull;
}

__global__ void k_seed_all(uint32_t n, uint32_t* list0, uint32_t* flag0, unsigned long long* key0,
                           unsigned long long* gmin, uint32_t* ctrl)
{
    uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    list0[q] = q;
    flag0[q] = kFull;
    key0[q] = 0ull;
    if (q == 0)
    {
        ctrl[kCtrlCount] = n;
        gmin[0] = 0ull;
    }
}

// seeds every tile of the given tile-row ranges (domain-decomposition resume)
__global__ void k_seed_rows(uint32_t ntx, const uint32_t* tile_rows, uint32_t n_tile_rows, uint32_t* list0,
                            uint32_t* flag0, unsigned long long* key0, unsigned long long* gmin,
                            uint32_t* ctrl)
{
    uint32_t n = n_tile_rows * ntx;
    uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    uint32_t tile_id = tile_rows[q / ntx] * ntx + q % ntx;
    flag0[tile_id] = kFull;
    key0[tile_id] = 0ull;
    list0[q] = tile_id;
    if (q == 0)
    {
        ctrl[kCtrlCount] = n;
        gmin[0] = 0ull;
    }
}

// adds every tile of the given tile rows to a list that may already hold pending tiles
__global__ void k_seed_rows_add(uint32_t ntx, const uint32_t* tile_rows, uint32_t n_tile_rows, uint32_t* list,
                                uint32_t* flag, unsigned long long* key, unsigned long long* gmin_cur,
                                uint32_t* count_cur, unsigned long long seed_key)
{
    uint32_t n = n_tile_rows * ntx;
    uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    uint32_t tile_id = tile_rows[q / ntx] * ntx + q % ntx;
    atomicMin(&key[tile_id], seed_key);
    if (atomicOr(&flag[tile_id], kFull) == 0) list[atomicAdd(count_cur, 1u)] = tile_id;
    if (q == 0) atomicMin(gmin_cur, seed_key);
}

__global__ void k_import_rows_min(double* T, uint32_t pitch, uint32_t nx, uint32_t j0, uint32_t n_rows,
                                  const double* src, int* changed, unsigned long long* min_lowered)
{
    size_t total = (size_t)nx * n_rows;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    int any = 0;
    unsigned long long lowest = kNoKey;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += stride)
    {
        uint32_t r = (uint32_t)(k / nx), i = (uint32_t)(k % nx);
        double v = src[k];
        double* t = &T[(size_t)(j0 + r) * pitch + i];
        if (v < *t)
        {
            *t = v;
            any = 1;
            lowest = min(lowest, key_of(v));
        }
    }
    if (__any_sync(0xffffffffu, any))
    {
        for (int o = 16; o > 0; o >>= 1) lowest = min(lowest, __shfl_xor_sync(0xffffffffu, lowest, o));
        if ((threadIdx.x & 31) == 0)
        {
            *changed = 1;
            atomicMin(min_lowered, lowest);
        }
    }
}

template <int MODE> int launch_fim(dymu_ctx* ctx, Params& prm, size_t total_tiles)
{
    constexpr size_t smem = (MODE == 2 || MODE == 4) ? SMEM_ANISO : SMEM;
    // persistent grid = every CTA that can be co-resident (required by the grid barrier)
    int per_sm = 0;
    DYMU_CUDA_TRY(ctx, cudaFuncSetAttribute(k_fim<MODE>,
                                            cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)smem));
    DYMU_CUDA_TRY(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(
                           &per_sm, k_fim<MODE>, THREADS, smem));
    if (per_sm < 1) DYMU_FAIL(ctx, DYMU_ERR_CUDA, "FIM kernel does not fit on an SM");
    size_t grid = (size_t)per_sm * ctx->sm_count;
    if (grid > total_tiles) grid = total_tiles;
    if (grid < 1) grid = 1;
    void* args[] = {&prm};
    DYMU_CUDA_TRY(ctx, cudaLaunchCooperativeKernel((void*)k_fim<MODE>, dim3((unsigned)grid),
                                                   dim3(THREADS), args,
                                                   smem, ctx->stream));
    ctx->launches++;
    return DYMU_OK;
}
}  // namespace

int dymu_internal_fim_alloc(dymu_ctx* ctx, dymu_fim_work* w, size_t capacity)
{
    dymu_internal_fim_free(w);
    w->capacity = capacity;
    for (int k = 0; k < 3; ++k)
    {
        DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&w->list[k], capacity * sizeof(uint32_t)));
        DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&w->flag[k], capacity * sizeof(uint32_t)));
        DYMU_CUDA_TRY(ctx, cudaMemsetAsync(w->flag[k], 0, capacity * sizeof(uint32_t), ctx->stream));
        DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&w->key[k], capacity * sizeof(unsigned long long)));
        DYMU_CUDA_TRY(ctx, cudaMemsetAsync(w->key[k], 0xFF, capacity * sizeof(unsigned long long),
                                           ctx->stream));
    }
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&w->ctrl, kCtrlWords * sizeof(uint32_t)));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&w->gmin, 4 * sizeof(unsigned long long)));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&w->dsave, capacity * sizeof(uint32_t)));
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(w->dsave, 0, capacity * sizeof(uint32_t), ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&w->stats, kStatWords * sizeof(unsigned long long)));
    w->rot = 0;
    w->pending = false;
    w->unclean = false;
    return DYMU_OK;
}

void dymu_internal_fim_free(dymu_fim_work* w)
{
    for (int k = 0; k < 3; ++k)
    {
        if (w->list[k]) cudaFree(w->list[k]);
        if (w->flag[k]) cudaFree(w->flag[k]);
        if (w->key[k]) cudaFree(w->key[k]);
        w->list[k] = w->flag[k] = nullptr;
        w->key[k] = nullptr;
    }
    if (w->ctrl) cudaFree(w->ctrl);
    if (w->gmin) cudaFree(w->gmin);
    if (w->dsave) cudaFree(w->dsave);
    w->gmin = nullptr;
    w->dsave = nullptr;
    if (w->stats) cudaFree(w->stats);
    w->ctrl = nullptr;
    w->stats = nullptr;
    w->capacity = 0;
}

int dymu_internal_fim_configure(dymu_ctx* ctx)
{
    int dev_coop = 0;
    DYMU_CUDA_TRY(ctx, cudaDeviceGetAttribute(&dev_coop, cudaDevAttrCooperativeLaunch, ctx->device));
    if (!dev_coop) DYMU_FAIL(ctx, DYMU_ERR_NODEVICE, "device lacks cooperative launch");
    ctx->fim_band = 1.0 / 0.0;  // until C_eff is first computed
    return DYMU_OK;
}

int dymu_internal_fim_clear(dymu_ctx* ctx, dymu_fim_work* w)
{
    DYMU_TRY(dymu_internal_settle_delivery(ctx));
    if (w->unclean)
    {
        // the previous launch did not drain its lists (phase-bounded solve that was abandoned,
        // NOCONV, failed launch): wake-up flags, keys and saved dirty masks may be set, and a set
        // flag would swallow the wake-up of that tile in this solve
        for (int k = 0; k < 3; ++k)
        {
            DYMU_CUDA_TRY(ctx, cudaMemsetAsync(w->flag[k], 0, w->capacity * sizeof(uint32_t), ctx->stream));
            DYMU_CUDA_TRY(ctx, cudaMemsetAsync(w->key[k], 0xFF, w->capacity * sizeof(unsigned long long),
                                               ctx->stream));
        }
        DYMU_CUDA_TRY(ctx, cudaMemsetAsync(w->dsave, 0, w->capacity * sizeof(uint32_t), ctx->stream));
    }
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(w->ctrl, 0, kCtrlWords * sizeof(uint32_t), ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(w->gmin, 0xFF, 4 * sizeof(unsigned long long), ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(w->stats, 0, kStatWords * sizeof(unsigned long long), ctx->stream));
    w->rot = 0;
    w->pending = false;
    return DYMU_OK;
}

int dymu_internal_fim_seed_maps(dymu_ctx* ctx, dymu_fim_work* w, const uint32_t* d_goal_ij, uint32_t n)
{
    DYMU_TRY(dymu_internal_fim_clear(ctx, w));
    k_seed_maps<<<1, 32, 0, ctx->stream>>>(ctx->T, (size_t)ctx->pitch * ctx->rows, ctx->pitch, ctx->ntx, ctx->nty,
                                           d_goal_ij, n, ctx->maps, w->list[0], w->flag[0], w->key[0], w->gmin,
                                           w->ctrl, w->stats);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    return DYMU_OK;
}

int dymu_internal_fim_seed_all(dymu_ctx* ctx, dymu_fim_work* w, uint32_t n_tiles)
{
    DYMU_TRY(dymu_internal_fim_clear(ctx, w));
    k_seed_all<<<dymu_div_up(n_tiles, 128), 128, 0, ctx->stream>>>(n_tiles, w->list[0], w->flag[0], w->key[0],
                                                                    w->gmin, w->ctrl);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    return DYMU_OK;
}

dymu_fim_launch dymu_internal_global_launch(dymu_ctx* ctx, uint32_t nprob)
{
    dymu_fim_launch L;
    L.T = ctx->T; L.slot_stride = (size_t)ctx->pitch * ctx->rows; L.C = ctx->ceff;
    L.pitch = ctx->pitch; L.rows = ctx->rows; L.ntx = ctx->ntx; L.nty = ctx->nty; L.nprob = nprob;
    L.work = &ctx->work;
    L.mode = ctx->aniso_n ? 2 : 0;
    L.A = ctx->aniso_n ? ctx->dircost : nullptr;
    L.band = ctx->aniso_n ? ctx->aniso_band : ctx->fim_band;
    return L;
}

// Runs the persistent kernel on the work lists as the caller left them and collects statistics.
int dymu_internal_fim_run(dymu_ctx* ctx, const dymu_fim_launch& L, dymu_solve_stats* stats)
{
    dymu_fim_work* w = L.work;
    Params prm;
    prm.T = L.T;
    prm.slot_stride = L.slot_stride;
    prm.C = L.C;
    prm.pitch = L.pitch;
    prm.rows = L.rows;
    prm.ntx = L.ntx;
    prm.nty = L.nty;
    prm.nprob = L.nprob;
    prm.list0 = w->list[0]; prm.list1 = w->list[1]; prm.list2 = w->list[2];
    prm.flag0 = w->flag[0]; prm.flag1 = w->flag[1]; prm.flag2 = w->flag[2];
    prm.key0 = w->key[0]; prm.key1 = w->key[1]; prm.key2 = w->key[2];
    prm.gmin = w->gmin;
    prm.dsave = w->dsave;
    prm.cta_trace = nullptr;
    prm.cta_trace_phases = 0;
    unsigned long long* d_cta_trace = nullptr;
    const uint32_t cta_trace_phases = 400;
    const char* cta_trace_path = getenv("DYMU_FIM_CTA_TRACE");
#ifdef DYMU_FIM_PROFILE
    if (cta_trace_path && L.mode == 0)
    {
        size_t bytes = (size_t)cta_trace_phases * 1024 * 8 * 8;
        DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&d_cta_trace, bytes));
        DYMU_CUDA_TRY(ctx, cudaMemsetAsync(d_cta_trace, 0, bytes, ctx->stream));
        prm.cta_trace = d_cta_trace;
        prm.cta_trace_phases = cta_trace_phases;
    }
#endif
    prm.ctrl = w->ctrl;
    prm.stats = w->stats;
    prm.stop_flag = L.stop_flag;
    prm.stop_value = L.stop_value;
    prm.tmax = nullptr;
    prm.xout = nullptr;
    prm.xld = 0;
    prm.xnx = ctx->nx;
    prm.xny = ctx->ny;
    prm.xminus1 = ctx->export_xform == DYMU_XFORM_INF_TO_MINUS1;
    if (L.mode != 1 && L.nprob == 1 && L.T == ctx->T && ctx->tile_tmax && (L.track_final || L.export_now))
    {
        prm.tmax = ctx->tile_tmax;
        if (L.export_now && ctx->export_dev)
        {
            prm.xout = ctx->export_dev;
            prm.xld = ctx->export_ld;
        }
    }
    prm.band = L.band;
    prm.A = L.A;
    prm.a_stride = L.slot_stride;
    // a wave needs at most ~(ntx+nty) tile hops in free space; obstacles lengthen the
    // geodesic, so leave two orders of magnitude of head room before reporting NOCONV
    prm.max_outer = 64 * (int)(L.ntx + L.nty) + 4096;
    if (L.max_phases > 0) prm.max_outer = (int)L.max_phases;
    const bool bounded = L.max_phases > 0 || L.stop_flag;
    prm.outer0 = w->rot;
    size_t total_tiles = (size_t)L.ntx * L.nty * L.nprob;
    w->unclean = true;  // until this launch reports that it drained its lists
    DYMU_CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    int rc;
    if ((L.mode == 2 || L.mode == 4) && !L.A)
        DYMU_FAIL(ctx, DYMU_ERR_STATE, "anisotropic solve without directional costs");
    rc = (L.mode == 0)   ? launch_fim<0>(ctx, prm, total_tiles)
         : (L.mode == 1) ? launch_fim<1>(ctx, prm, total_tiles)
         : (L.mode == 2) ? launch_fim<2>(ctx, prm, total_tiles)
         : (L.mode == 3) ? launch_fim<3>(ctx, prm, total_tiles)
                         : launch_fim<4>(ctx, prm, total_tiles);
    DYMU_TRY(rc);
    DYMU_CUDA_TRY(ctx, cudaEventRecord(ctx->ev2, ctx->stream));
    if (prm.xout)
    {
        // the tiles that are left go out on the copy stream, beside whatever follows on the main one
        DYMU_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev2, 0));
        const uint32_t nt = L.ntx * L.nty;
        const uint32_t g = nt < (uint32_t)ctx->sm_count * 2 ? nt : (uint32_t)ctx->sm_count * 2;
        k_deliver_rest<<<g, 512, 0, ctx->copy_stream>>>(prm.T, prm.pitch, prm.ntx, prm.nty, prm.tmax, prm.xout,
                                                        prm.xld, prm.xnx, prm.xny, prm.xminus1, prm.stats);
        ctx->launches++;
        DYMU_CUDA_TRY(ctx, cudaGetLastError());
        DYMU_CUDA_TRY(ctx, cudaEventRecord(ctx->ev_tail, ctx->copy_stream));
        ctx->export_tail_pending = true;
    }
    unsigned long long h[kStatWords];
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(h, w->stats, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    const bool converged = h[kStatConverged] != 0;
    const uint32_t delivered = (uint32_t)h[kStatDelivered];
#ifdef DYMU_FIM_PROFILE
    if (L.mode == 0)
    {
        const double fetch = h[kStatCycFetch], load = h[kStatCycLoad], sweep = h[kStatCycSweep],
                     store = h[kStatCycStore], barrier = h[kStatCycBarrier], tiles = h[kStatTiles];
        const double tot = fetch + load + sweep + store + barrier;
        fprintf(stderr, "[fim profile] cycles/CTA-sum: fetch %.1f%% load %.1f%% sweep %.1f%% store %.1f%% barrier %.1f%%;"
                " per activation: load %.0f sweep %.0f store %.0f cyc; per sweep %.0f cyc; fetch+barrier per CTA-phase %.0f cyc\n",
                100 * fetch / tot, 100 * load / tot, 100 * sweep / tot, 100 * store / tot, 100 * barrier / tot,
                load / tiles, sweep / tiles, store / tiles, sweep / (h[kStatSweeps] ? h[kStatSweeps] : 1),
                (fetch + barrier) / ((double)h[kStatPhases] * 444));
    }
#endif
    if (d_cta_trace)
    {
        size_t bytes = (size_t)cta_trace_phases * 1024 * 8 * 8;
        void* hb = malloc(bytes);
        cudaMemcpy(hb, d_cta_trace, bytes, cudaMemcpyDeviceToHost);
        if (FILE* f = fopen(cta_trace_path, "wb"))
        {
            fwrite(hb, 1, bytes, f);
            fclose(f);
        }
        free(hb);
        cudaFree(d_cta_trace);
    }
    if (stats)
    {
        stats->tile_activations = h[kStatTiles];
        stats->cell_updates = h[kStatVisits] * 32ull;  // n_visits counts 32-cell warp evaluations
        stats->outer_iterations = (uint32_t)h[kStatPhases];
        stats->converged = converged;
        stats->tiles_deferred = h[kStatDeferred];
        stats->inner_iterations = h[kStatSweeps];
        stats->goal_obstacle = (uint32_t)h[kStatGoalObstacle];
        stats->cells_written = h[kStatWritten];
        stats->tiles_delivered_early = delivered;
        // (k_deliver_rest is still running: counted from here)
        const uint32_t nt_all = L.ntx * L.nty;
        stats->tiles_delivered_late = (prm.xout && converged && nt_all > delivered) ? nt_all - delivered : 0;
        DYMU_CUDA_TRY(ctx, cudaEventElapsedTime(&stats->kernel_ms, ctx->ev1, ctx->ev2));
    }
    if (h[kStatAbort])
    {
        // a CTA waited eight seconds at the grid barrier and the grid gave up (see barrier_spin)
        w->pending = false;
        DYMU_FAIL(ctx, DYMU_ERR_CUDA, "tile FIM: the grid barrier timed out after %llu phases (solver defect); "
                                      "the total-cost plane is not valid", h[kStatPhases]);
    }
    if (prm.xout && converged) ctx->export_done = true;  // the tail ran: the caller's matrix is complete
    w->rot = (int)((prm.outer0 + h[kStatPhases]) % 3);
    w->pending = !converged;
    w->unclean = !converged;
    if (!converged && !bounded)
        DYMU_FAIL(ctx, DYMU_ERR_NOCONV, "tile FIM hit the outer-iteration cap (%d) before converging",
                  prm.max_outer);
    return DYMU_OK;
}

int dymu_internal_fill(dymu_ctx* ctx, double* p, double v, size_t n);

namespace
{
__global__ void k_selftest_sqrt(unsigned long long seed, unsigned long long n, unsigned long long* bad,
                                double* first_bad)
{
    unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long k = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride)
    {
        // splitmix64 -> mantissa + an exponent spread over 2^-120 .. 2^120
        unsigned long long z = seed + (k + 1) * 0x9E3779B97F4A7C15ull;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        z ^= z >> 31;
        unsigned long long mant = z & 0x000FFFFFFFFFFFFFull;
        unsigned long long ex = 1023ull - 120ull + ((z >> 52) % 241ull);
        double x = __longlong_as_double((long long)((ex << 52) | mant));
        if ((k & 7) == 0) x = (double)((z >> 40) & 0xFFFFFF) * (double)((z >> 40) & 0xFFFFFF) + 0.0;  // perfect squares
        if (x <= 0) x = 1.0;
        double a = dymu_sqrt_normal(x), b = sqrt(x);
        if (__double_as_longlong(a) != __double_as_longlong(b))
            if (atomicAdd(bad, 1ull) == 0) *first_bad = x;
    }
}
}  // namespace

extern "C" {

int dymu_selftest_sqrt(dymu_ctx* ctx, uint64_t n, uint64_t seed, uint64_t* mismatches, double* first_bad)
{
    DYMU_GUARD(ctx);
    if (!ctx || !mismatches) return DYMU_ERR_ARG;
    unsigned long long* d = (unsigned long long*)ctx->d_scratch;
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(d, 0, 16, ctx->stream));
    k_selftest_sqrt<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(seed, n, d, (double*)(d + 1));
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    unsigned long long h[2];
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(h, d, 16, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *mismatches = h[0];
    if (first_bad) memcpy(first_bad, &h[1], 8);
    return DYMU_OK;
}

int dymu_reserve_slots(dymu_ctx* ctx, uint32_t n_slots)
{
    DYMU_GUARD(ctx);
    if (!ctx || n_slots < 1) return DYMU_ERR_ARG;
    if (n_slots == ctx->n_slots) return DYMU_OK;
    size_t n = (size_t)ctx->pitch * ctx->rows;
    double* T = nullptr;
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&T, n * n_slots * sizeof(double)));
    cudaFree(ctx->T);
    ctx->T = T;
    ctx->n_slots = n_slots;
    DYMU_TRY(dymu_internal_fill(ctx, ctx->T, 1.0 / 0.0, n * n_slots));
    DYMU_TRY(dymu_internal_fim_alloc(ctx, &ctx->work, (size_t)ctx->ntx * ctx->nty * n_slots));
    dymu_internal_unmark_all(ctx);
    ctx->solved = false;
    return DYMU_OK;
}

static int solve_total_cost_impl(dymu_ctx* ctx, uint32_t n_goals, const uint32_t* goal_i,
                                 const uint32_t* goal_j, uint32_t max_phases, uint32_t stop_value,
                                 dymu_solve_stats* stats)
{
    if (!ctx || !goal_i || !goal_j || n_goals < 1 || n_goals > ctx->n_slots) return DYMU_ERR_ARG;
    if (!ctx->have_cost) DYMU_FAIL(ctx, DYMU_ERR_STATE, "no cost map: call dymu_set_cost_map / dymu_compute_cost_map first");
    for (uint32_t q = 0; q < n_goals; ++q)
        if (goal_i[q] >= ctx->nx || goal_j[q] >= ctx->ny) DYMU_FAIL(ctx, DYMU_ERR_ARG, "goal %u outside the grid", q);
    DYMU_TRY(dymu_internal_refresh_ceff(ctx));
    DYMU_TRY(dymu_internal_settle_delivery(ctx));
    size_t n = (size_t)ctx->pitch * ctx->rows;
    // resetTotalCostMap, G.cpp:473-485 (whole plane instead of the propagated-node list)
    DYMU_CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    DYMU_TRY(dymu_internal_fill(ctx, ctx->T, 1.0 / 0.0, n * n_goals));
    dymu_internal_unmark_slots(ctx, 0, n_goals);
    DYMU_TRY(dymu_internal_scratch(ctx, (size_t)n_goals * 8, (size_t)n_goals * 8));
    uint32_t* h_goals = (uint32_t*)ctx->h_pinned;
    for (uint32_t q = 0; q < n_goals; ++q)
    {
        h_goals[2 * q] = goal_i[q];
        h_goals[2 * q + 1] = goal_j[q];
    }
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_scratch, h_goals, (size_t)n_goals * 8,
                                       cudaMemcpyHostToDevice, ctx->stream));
    dymu_fim_launch L = dymu_internal_global_launch(ctx, n_goals);
    L.max_phases = max_phases;
    L.stop_flag = stop_value ? ctx->d_upflag : nullptr;
    L.stop_value = stop_value;
    ctx->export_done = false;
    if (ctx->export_dev && n_goals == 1)
    {
        // direct delivery: every tile starts as "not finished" (+inf)
        const size_t nt = (size_t)ctx->ntx * ctx->nty;
        if (ctx->tile_tmax_cap < nt)
        {
            if (ctx->tile_tmax) cudaFree(ctx->tile_tmax);
            ctx->tile_tmax = nullptr;
            ctx->tile_tmax_cap = 0;
            DYMU_CUDA_TRY(ctx, cudaMalloc((void**)&ctx->tile_tmax, nt * sizeof(unsigned long long)));
            ctx->tile_tmax_cap = nt;
        }
        DYMU_TRY(dymu_internal_fill(ctx, (double*)ctx->tile_tmax, 1.0 / 0.0, nt));
        L.track_final = true;
        // a phase-bounded launch is the head of a streamed solve: cost rows are still missing, and
        // values that look finished may still drop when they arrive
        L.export_now = (max_phases == 0);
    }
    dymu_fim_work* w = &ctx->work;
    DYMU_TRY(dymu_internal_fim_clear(ctx, w));
    k_seed<<<1, 32, 0, ctx->stream>>>(ctx->T, n, ctx->pitch, ctx->ntx, ctx->nty, TILE,
                                      (const uint32_t*)ctx->d_scratch, n_goals, ctx->obst, w->list[0],
                                      w->flag[0], w->key[0], w->gmin, w->ctrl, w->stats);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    dymu_solve_stats local;
    memset(&local, 0, sizeof(local));
    int rc = dymu_internal_fim_run(ctx, L, &local);
    if (rc == DYMU_OK || rc == DYMU_ERR_NOCONV)
    {
        cudaEventElapsedTime(&local.reset_ms, ctx->ev0, ctx->ev1);
        if (stats) *stats = local;
    }
    ctx->solved = (rc == DYMU_OK) && local.converged;
    ctx->last_n_goals = n_goals;
    ctx->last_goal_i = goal_i[0];
    ctx->last_goal_j = goal_j[0];
    return rc;
}

static int solve_streamed(dymu_ctx* ctx, uint32_t goal_i, uint32_t goal_j, uint32_t first_phases,
                          dymu_solve_stats* stats);

int dymu_solve_total_cost(dymu_ctx* ctx, uint32_t n_goals, const uint32_t* goal_i,
                          const uint32_t* goal_j, dymu_solve_stats* stats)
{
    DYMU_GUARD_ONLY(ctx);
    if (ctx && ctx->upload_pending)
    {
        // a cost map is still on its way (dymu_set_cost_map_begin): start on the rows that are there
        // (the anisotropic solve waits for the whole map: its directional costs need every row; so
        // does obstacle clearance, which near a seam needs obstacles of rows still on their way)
        if (!ctx->aniso_n && !ctx->clear_on && n_goals == 1 && goal_i && goal_j && goal_i[0] < ctx->nx && goal_j[0] >= ctx->up_a0
            && goal_j[0] < ctx->up_a1)
            return solve_streamed(ctx, goal_i[0], goal_j[0], 0, stats);
        DYMU_TRY(dymu_internal_settle_upload(ctx));
    }
    return solve_total_cost_impl(ctx, n_goals, goal_i, goal_j, 0, 0, stats);
}

int dymu_solve_start(dymu_ctx* ctx, uint32_t goal_i, uint32_t goal_j, uint32_t max_phases,
                     dymu_solve_stats* stats)
{
    DYMU_GUARD(ctx);
    if (max_phases == 0) return DYMU_ERR_ARG;
    if (ctx && ctx->aniso_n) DYMU_FAIL(ctx, DYMU_ERR_STATE, "phase-bounded solves are isotropic only");
    return solve_total_cost_impl(ctx, 1, &goal_i, &goal_j, max_phases, 0, stats);
}

static int solve_resume_impl(dymu_ctx* ctx, const uint32_t* ranges, uint32_t n_ranges, double seed_key,
                             uint32_t max_phases, uint32_t stop_value, dymu_solve_stats* stats,
                             bool deliver = false)
{
    if (!ctx || (!ranges && n_ranges)) return DYMU_ERR_ARG;
    if (!deliver) ctx->export_done = false;
    if (!ctx->have_cost) DYMU_FAIL(ctx, DYMU_ERR_STATE, "no cost map");
    if (n_ranges == 0 && !ctx->work.pending)
    {
        // nothing queued and nothing new: the plane is at its fixed point
        if (stats)
        {
            memset(stats, 0, sizeof(*stats));
            stats->converged = 1;
        }
        return DYMU_OK;
    }
    for (uint32_t k = 0; k < n_ranges; ++k)
        if (ranges[2 * k] >= ranges[2 * k + 1] || ranges[2 * k + 1] > ctx->ny) return DYMU_ERR_ARG;
    DYMU_TRY(dymu_internal_refresh_ceff(ctx));
    DYMU_TRY(dymu_internal_settle_delivery(ctx));
    dymu_internal_unmark_slots(ctx, 0, 1);
    // distinct tile rows covered by the ranges
    DYMU_TRY(dymu_internal_scratch(ctx, sizeof(uint32_t) * ctx->nty, sizeof(uint32_t) * ctx->nty));
    uint32_t* h_rows = (uint32_t*)ctx->h_pinned;
    uint32_t n_rows = 0;
    for (uint32_t ty = 0; ty < ctx->nty; ++ty)
    {
        bool hit = false;
        for (uint32_t k = 0; k < n_ranges && !hit; ++k)
            hit = (ranges[2 * k] < (ty + 1) * kTile) && (ranges[2 * k + 1] > ty * kTile);
        if (hit) h_rows[n_rows++] = ty;
    }
    const uint32_t* d_rows = (const uint32_t*)ctx->d_scratch;
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_scratch, h_rows, sizeof(uint32_t) * n_rows, cudaMemcpyHostToDevice,
                                       ctx->stream));
    dymu_fim_work* w = &ctx->work;
    if (w->pending)
    {
        // continue with the lists the previous launch left behind; the rows are merged in at seed_key.
        // Only the barrier counter and the stop request (kCtrlBarrier, kCtrlStopAt) start again.
        const int cur = w->rot;
        DYMU_CUDA_TRY(ctx, cudaMemsetAsync(w->ctrl + kCtrlBarrier, 0, (kCtrlWords - kCtrlBarrier) * sizeof(uint32_t),
                                           ctx->stream));
        DYMU_CUDA_TRY(ctx, cudaMemsetAsync(w->stats, 0, kStatWords * sizeof(unsigned long long), ctx->stream));
        if (n_rows)
            k_seed_rows_add<<<dymu_div_up(n_rows * ctx->ntx, 128), 128, 0, ctx->stream>>>(
                ctx->ntx, d_rows, n_rows, w->list[cur], w->flag[cur], w->key[cur], w->gmin + cur,
                w->ctrl + kCtrlCount + cur, (unsigned long long)__builtin_bit_cast(long long, seed_key));
    }
    else
    {
        DYMU_TRY(dymu_internal_fim_clear(ctx, w));
        if (n_rows)
            k_seed_rows<<<dymu_div_up(n_rows * ctx->ntx, 128), 128, 0, ctx->stream>>>(
                ctx->ntx, d_rows, n_rows, w->list[0], w->flag[0], w->key[0], w->gmin, w->ctrl);
    }
    if (n_rows)
    {
        ctx->launches++;
        DYMU_CUDA_TRY(ctx, cudaGetLastError());
    }
    dymu_fim_launch L = dymu_internal_global_launch(ctx, 1);
    L.max_phases = max_phases;
    L.stop_flag = stop_value ? ctx->d_upflag : nullptr;
    L.stop_value = stop_value;
    // the tail of a streamed solve: the whole cost map is there now (tile bounds were tracked by the head)
    L.track_final = ctx->export_dev && ctx->tile_tmax;  // (values only drop: older bounds stay valid)
    L.export_now = deliver && L.track_final && max_phases == 0;
    dymu_solve_stats local;
    memset(&local, 0, sizeof(local));
    const int rc = dymu_internal_fim_run(ctx, L, &local);
    if (stats && (rc == DYMU_OK || rc == DYMU_ERR_NOCONV)) *stats = local;
    return rc;
}

int dymu_solve_advance(dymu_ctx* ctx, const uint32_t* ranges, uint32_t n_ranges, double seed_key,
                       uint32_t max_phases, dymu_solve_stats* stats)
{
    DYMU_GUARD(ctx);
    if (max_phases == 0 || !(seed_key >= 0.0)) return DYMU_ERR_ARG;
    if (ctx && ctx->aniso_n) DYMU_FAIL(ctx, DYMU_ERR_STATE, "phase-bounded solves are isotropic only");
    return solve_resume_impl(ctx, ranges, n_ranges, seed_key, max_phases, 0, stats);
}

int dymu_set_cost_map_begin(dymu_ctx* ctx, const double* cost_host, size_t ld, uint32_t first_row)
{
    DYMU_GUARD_ONLY(ctx);
    if (!ctx || !cost_host || ld < ctx->nx) return DYMU_ERR_ARG;
    if (ctx->upload_pending) DYMU_TRY(dymu_internal_settle_upload(ctx));
    if (first_row >= ctx->ny) first_row = ctx->ny / 2;
    const uint32_t ny = ctx->ny;
    // Three parts, nearest first: a thin band of rows around `first_row` (the solve starts as soon
    // as it is there), a wider band around it, everything else.  Behind the second and the third
    // part the copy engine writes 1 / 2 into a device word the running solve kernel looks at.
    auto band = [&](uint32_t reach, uint32_t& r0, uint32_t& r1) {
        r0 = first_row > reach ? ((first_row - reach) / kTile) * kTile : 0;
        r1 = first_row + reach < ny ? dymu_div_up(first_row + reach, kTile) * kTile : ny;
        if (r1 > ny) r1 = ny;
    };
    uint32_t a0, a1, b0, b1;
    band(4 * kTile, a0, a1);
    band(ny / 8 < 256 ? 256 : ny / 8, b0, b1);
    if (b0 > a0) b0 = a0;
    if (b1 < a1) b1 = a1;
    auto h2d_rows = [&](uint32_t j0, uint32_t j1) -> int {
        if (j0 >= j1) return DYMU_OK;
        DYMU_CUDA_TRY(ctx, cudaMemcpy2DAsync(ctx->cost + (size_t)j0 * ctx->pitch, ctx->pitch * sizeof(double),
                                             cost_host + (size_t)j0 * ld, ld * sizeof(double),
                                             ctx->nx * sizeof(double), j1 - j0, cudaMemcpyHostToDevice,
                                             ctx->copy_stream));
        return DYMU_OK;
    };
    auto flag = [&](uint32_t v) -> int {
        DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_upflag, ctx->h_upvals + v, sizeof(uint32_t),
                                           cudaMemcpyHostToDevice, ctx->copy_stream));
        return DYMU_OK;
    };
    // the copies must not overtake earlier work on the planes (a previous plan's read-back)
    DYMU_CUDA_TRY(ctx, cudaEventRecord(ctx->ev_up, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_up, 0));
    DYMU_TRY(flag(0));
    DYMU_TRY(h2d_rows(a0, a1));
    DYMU_CUDA_TRY(ctx, cudaEventRecord(ctx->ev_part0, ctx->copy_stream));
    DYMU_TRY(h2d_rows(b0, a0));
    DYMU_TRY(h2d_rows(a1, b1));
    DYMU_TRY(flag(1));
    DYMU_CUDA_TRY(ctx, cudaEventRecord(ctx->ev_part, ctx->copy_stream));
    DYMU_TRY(h2d_rows(0, b0));
    DYMU_TRY(h2d_rows(b1, ny));
    DYMU_TRY(flag(2));
    DYMU_CUDA_TRY(ctx, cudaEventRecord(ctx->ev_up, ctx->copy_stream));
    ctx->upload_pending = true;
    ctx->up_a0 = a0;
    ctx->up_a1 = a1;
    ctx->up_b0 = b0;
    ctx->up_b1 = b1;
    ctx->solved = false;
    return DYMU_OK;
}

// the work counters and the kernel time of one more launch of the same solve
static void add_work(dymu_solve_stats* s, const dymu_solve_stats& p)
{
    s->outer_iterations += p.outer_iterations;
    s->tile_activations += p.tile_activations;
    s->cell_updates += p.cell_updates;
    s->tiles_deferred += p.tiles_deferred;
    s->inner_iterations += p.inner_iterations;
    s->cells_written += p.cells_written;
    s->kernel_ms += p.kernel_ms;
}

// The solve of a cost map whose upload (dymu_set_cost_map_begin) is still in flight.  The rows that
// have arrived are opened, the rest stays impassable (C_eff = +inf); the kernel hands back when the
// copy engine reports the next part (or after `first_phases` phases when the caller fixes the cut),
// that part is opened, the tiles along its seams are woken, and the solve goes on from its work lists.
static int solve_streamed(dymu_ctx* ctx, uint32_t goal_i, uint32_t goal_j, uint32_t first_phases,
                          dymu_solve_stats* stats)
{
    const uint32_t a0 = ctx->up_a0, a1 = ctx->up_a1, b0 = ctx->up_b0, b1 = ctx->up_b1, ny = ctx->ny;
    ctx->upload_pending = false;
    // DYMU_STREAM_PHASES=n: cut the launches after n / 2n phases instead of on the copy engine's word
    if (first_phases == 0)
        if (const char* e = getenv("DYMU_STREAM_PHASES"))
            if (atoi(e) > 0) first_phases = (uint32_t)atoi(e);
    // everything not uploaded yet is impassable for now
    DYMU_TRY(dymu_internal_fill(ctx, ctx->ceff, 1.0 / 0.0, (size_t)ctx->pitch * ctx->rows));
    DYMU_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_part0, 0));
    DYMU_TRY(dymu_internal_cost_rows(ctx, a0, a1));
    ctx->have_cost = true;
    ctx->ceff_dirty = false;
    // band width of the scheduler from the rows that are there (the mean cost of a Mars-like map
    // does not change much from one band of rows to the next)
    DYMU_TRY(dymu_internal_band_from_rows(ctx, a0, a1));
    dymu_solve_stats part[3];
    memset(part, 0, sizeof(part));
    // ---- part 1: until the second part is there
    int rc = solve_total_cost_impl(ctx, 1, &goal_i, &goal_j, first_phases ? first_phases : (1u << 20),
                                   first_phases ? 0 : 1, &part[0]);
    auto open_rows = [&](uint32_t lo0, uint32_t lo1, uint32_t hi0, uint32_t hi1, uint32_t* ranges,
                         uint32_t& n_ranges) -> int {
        // rows [lo0, lo1) below and [hi0, hi1) above what is open: C_eff, and the seam rows to wake
        n_ranges = 0;
        if (lo1 > lo0)
        {
            DYMU_TRY(dymu_internal_cost_rows(ctx, lo0, lo1));
            ranges[2 * n_ranges] = lo1 - 1;
            ranges[2 * n_ranges + 1] = lo1 + 1;
            n_ranges++;
        }
        if (hi1 > hi0)
        {
            DYMU_TRY(dymu_internal_cost_rows(ctx, hi0, hi1));
            ranges[2 * n_ranges] = hi0 - 1;
            ranges[2 * n_ranges + 1] = hi0 + 1;
            n_ranges++;
        }
        return DYMU_OK;
    };
    uint32_t ranges[4], n_ranges = 0;
    // ---- part 2: the wider band, until everything is there
    DYMU_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_part, 0));
    DYMU_TRY(open_rows(b0, a0, a1, b1, ranges, n_ranges));
    const bool seeded = rc == DYMU_OK && !part[0].goal_obstacle;
    if (seeded && (n_ranges || !part[0].converged))
    {
        const bool all_there = cudaEventQuery(ctx->ev_up) == cudaSuccess;
        cudaGetLastError();  // (cudaErrorNotReady is an answer, not a failure)
        if (!all_there || first_phases)
        {
            rc = solve_resume_impl(ctx, ranges, n_ranges, 0.0, first_phases ? 2 * first_phases : (1u << 20),
                                   first_phases ? 0 : 2, &part[1]);
            n_ranges = 0;
        }
    }
    else
        part[1].converged = part[0].converged;
    // ---- part 3: the rest, to the end
    DYMU_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_up, 0));
    uint32_t ranges3[8], n3 = 0;
    DYMU_TRY(open_rows(0, b0, b1, ny, ranges3, n3));
    for (uint32_t k = 0; k < n_ranges; ++k)  // seams of part 2 that were not woken yet
    {
        ranges3[2 * n3] = ranges[2 * k];
        ranges3[2 * n3 + 1] = ranges[2 * k + 1];
        n3++;
    }
    if (rc != DYMU_OK) return rc;
    if (part[0].goal_obstacle)
    {
        // nothing was seeded (G.cpp:447-451: "The goal is not valid"); the planes are complete
        if (stats) *stats = part[0];
        ctx->solved = false;
        return DYMU_OK;
    }
    if (n3 || ctx->work.pending)
        rc = solve_resume_impl(ctx, ranges3, n3, 0.0, 0, 0, &part[2], true);
    else
        part[2].converged = 1;
    if (stats)
    {
        *stats = part[0];
        add_work(stats, part[1]);
        add_work(stats, part[2]);
        stats->converged = part[2].converged;
        stats->tiles_delivered_early = part[2].tiles_delivered_early;
        stats->tiles_delivered_late = part[2].tiles_delivered_late;
    }
    ctx->solved = (rc == DYMU_OK);
    return rc;
}

int dymu_plan_streamed(dymu_ctx* ctx, const double* cost_host, size_t ld, uint32_t goal_i, uint32_t goal_j,
                       uint32_t first_phases, dymu_solve_stats* stats)
{
    DYMU_GUARD_ONLY(ctx);
    if (!ctx || !cost_host || ld < ctx->nx || goal_i >= ctx->nx || goal_j >= ctx->ny) return DYMU_ERR_ARG;
    DYMU_TRY(dymu_set_cost_map_begin(ctx, cost_host, ld, goal_j));
    if (ctx->aniso_n || ctx->clear_on)
    {
        // the directional costs and the clearance need the whole map: upload first, then the full solve
        DYMU_TRY(dymu_internal_settle_upload(ctx));
        return solve_total_cost_impl(ctx, 1, &goal_i, &goal_j, 0, 0, stats);
    }
    return solve_streamed(ctx, goal_i, goal_j, first_phases, stats);
}

int dymu_reset_total_cost(dymu_ctx* ctx)
{
    DYMU_GUARD(ctx);
    if (!ctx) return DYMU_ERR_ARG;
    DYMU_TRY(dymu_internal_settle_delivery(ctx));
    ctx->solved = false;
    ctx->export_done = false;
    ctx->work.pending = false;
    dymu_internal_unmark_slots(ctx, 0, 1);
    return dymu_internal_fill(ctx, ctx->T, 1.0 / 0.0, (size_t)ctx->pitch * ctx->rows);
}

int dymu_export_rows(dymu_ctx* ctx, uint32_t slot, uint32_t j0, uint32_t n_rows, double* dst,
                     int device_ptr)
{
    DYMU_GUARD(ctx);
    if (!ctx || !dst || slot >= ctx->n_slots || n_rows == 0 || (uint64_t)j0 + n_rows > ctx->ny)
        return DYMU_ERR_ARG;
    const double* src = ctx->T + (size_t)slot * ctx->pitch * ctx->rows + (size_t)j0 * ctx->pitch;
    DYMU_CUDA_TRY(ctx, cudaMemcpy2DAsync(dst, ctx->nx * sizeof(double), src, ctx->pitch * sizeof(double),
                                         ctx->nx * sizeof(double), n_rows,
                                         device_ptr ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost,
                                         ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DYMU_OK;
}

int dymu_import_rows_min_key(dymu_ctx* ctx, uint32_t slot, uint32_t j0, uint32_t n_rows,
                             const double* src, int device_ptr, int* changed, double* min_lowered)
{
    DYMU_GUARD(ctx);
    if (!ctx || !src || !changed || !min_lowered || slot >= ctx->n_slots || n_rows == 0
        || (uint64_t)j0 + n_rows > ctx->ny)
        return DYMU_ERR_ARG;
    DYMU_TRY(dymu_internal_settle_delivery(ctx));
    dymu_internal_unmark_slots(ctx, slot, 1);
    size_t bytes = (size_t)ctx->nx * n_rows * sizeof(double);
    DYMU_TRY(dymu_internal_scratch(ctx, bytes + 64, device_ptr ? 64 : bytes + 64));
    int* d_flag = (int*)ctx->d_scratch;
    unsigned long long* d_min = (unsigned long long*)((char*)ctx->d_scratch + 8);
    const double* d_src = src;
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(d_flag, 0, 8, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaMemsetAsync(d_min, 0xFF, 8, ctx->stream));
    if (!device_ptr)
    {
        double* stage = (double*)((char*)ctx->d_scratch + 64);
        memcpy((char*)ctx->h_pinned + 64, src, bytes);
        DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(stage, (char*)ctx->h_pinned + 64, bytes, cudaMemcpyHostToDevice,
                                           ctx->stream));
        d_src = stage;
    }
    size_t total = (size_t)ctx->nx * n_rows;
    int grid = (int)((total + 255) / 256);
    if (grid > ctx->sm_count * 8) grid = ctx->sm_count * 8;
    k_import_rows_min<<<grid, 256, 0, ctx->stream>>>(ctx->T + (size_t)slot * ctx->pitch * ctx->rows,
                                                     ctx->pitch, ctx->nx, j0, n_rows, d_src, d_flag, d_min);
    ctx->launches++;
    DYMU_CUDA_TRY(ctx, cudaGetLastError());
    unsigned long long h[2] = {0, 0};
    DYMU_CUDA_TRY(ctx, cudaMemcpyAsync(h, d_flag, 16, cudaMemcpyDeviceToHost, ctx->stream));
    DYMU_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *changed = (int)(h[0] & 0xffffffffu);
    if (*changed) ctx->solved = ctx->export_done = false;  // the plane moved away from the last solve's fixed point
    long long bits = (long long)h[1];
    double v;
    memcpy(&v, &bits, sizeof(v));
    *min_lowered = *changed ? v : 1.0 / 0.0;
    return DYMU_OK;
}

int dymu_stop_threshold(dymu_ctx* ctx, uint32_t slot, uint32_t start_i, uint32_t start_j,
                        double* t_stop)
{
    DYMU_GUARD(ctx);
    if (!ctx || !t_stop || slot >= ctx->n_slots) return DYMU_ERR_ARG;
    if (start_i < 1 || start_j < 1 || start_i + 1 >= ctx->nx || start_j + 1 >= ctx->ny)
        return DYMU_ERR_ARG;
    uint32_t idx[5] = {start_j * ctx->nx + start_i, (start_j - 1) * ctx->nx + start_i,
                       start_j * ctx->nx + start_i - 1, start_j * ctx->nx + start_i + 1,
                       (start_j + 1) * ctx->nx + start_i};
    double v[5];
    DYMU_TRY(dymu_read_cells(ctx, DYMU_PLANE_TOTAL_COST, slot, idx, 5, v));
    double m = v[0];
    for (int k = 1; k < 5; ++k)
        if (v[k] > m) m = v[k];
    *t_stop = m;
    return DYMU_OK;
}

}  // extern "C"
