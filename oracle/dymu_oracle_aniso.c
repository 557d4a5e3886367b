/* dymu_oracle_aniso.c -- plain-C restatement of the slope-anisotropic total-cost solve and
 * descent (dymu_set_anisotropy, DESIGN.md section 10).  Test infrastructure only: built into its
 * own library by oracle/oracle_aniso.py, never linked into the product.
 *
 * The translation unit includes the isotropic restatement (dymu_oracle.c) for its binary heap, the
 * per-axis rule of gradientNode (grad_axis) and interpolate (interp), so that the descent shares
 * that arithmetic with the isotropic one.
 *
 * Planes are dense [j][i] (nx * ny doubles each); the four directional-cost planes are stored
 * one after the other in the order i-1, i+1, j-1, j+1.  Every expression is written in the order
 * the device uses (no FMA contraction, correctly rounded sqrt and division). */
#include "dymu_oracle.c"

/* f(theta): piecewise linear in the table, clamped at both ends */
static double aniso_factor(const double* th, const double* f, int n, double t)
{
    if (t <= th[0]) return f[0];
    if (t >= th[n - 1]) return f[n - 1];
    int k = 0;
    while (t >= th[k + 1]) ++k;
    return f[k] + (f[k + 1] - f[k]) * ((t - th[k]) / (th[k + 1] - th[k]));
}

/* a(x->m) = C_eff(x) * f(atan((elev[m] - elev[x]) / gres) * (180/pi)); +inf where C_eff is +inf
 * and toward a neighbour outside the grid.  libm's atan. */
void orc_aniso_dircost(const double* elev, const double* ceff, uint32_t nx, uint32_t ny, double gres,
                       const double* th, const double* f, int n, double* A)
{
    const double kDeg = 180.0 / 3.141592653589793;
    const size_t plane = (size_t)nx * ny;
    for (uint32_t j = 0; j < ny; ++j)
        for (uint32_t i = 0; i < nx; ++i)
        {
            const size_t q = (size_t)j * nx + i;
            const double c = ceff[q];
            double a[4] = {ORC_INF, ORC_INF, ORC_INF, ORC_INF};
            if (c < ORC_INF)
            {
                const int has[4] = {i > 0, i + 1 < nx, j > 0, j + 1 < ny};
                const int64_t off[4] = {-1, 1, -(int64_t)nx, (int64_t)nx};
                for (int d = 0; d < 4; ++d)
                    if (has[d]) a[d] = c * aniso_factor(th, f, n, atan((elev[q + off[d]] - elev[q]) / gres) * kDeg);
            }
            for (int d = 0; d < 4; ++d) A[d * plane + q] = a[d];
        }
}

/* two-sided value of one neighbour pair (k_fim's aniso_pair) */
static double aniso_pair(double Th, double ah, double Tv, double av)
{
    const double d = Th - Tv;
    const double ah2 = ah * ah, av2 = av * av;
    const double s = ah2 + av2;
    if (!((d > -ah) && (d < av) && (s < ORC_INF))) return ORC_INF;
    return ((av2 * Th + ah2 * Tv) + (ah * av) * sqrt(s - d * d)) / s;
}

/* the anisotropic update of cell q (k_fim's relax_aniso) on the values of T */
static double aniso_update(const double* A, const double* T, uint32_t nx, uint32_t ny, size_t q)
{
    const size_t plane = (size_t)nx * ny;
    const uint32_t i = (uint32_t)(q % nx), j = (uint32_t)(q / nx);
    const double txm = i > 0 ? T[q - 1] : ORC_INF, txp = i + 1 < nx ? T[q + 1] : ORC_INF;
    const double tym = j > 0 ? T[q - nx] : ORC_INF, typ = j + 1 < ny ? T[q + nx] : ORC_INF;
    const double axm = A[q], axp = A[plane + q], aym = A[2 * plane + q], ayp = A[3 * plane + q];
    double t = fmin(fmin(txm + axm, txp + axp), fmin(tym + aym, typ + ayp));
    t = fmin(t, fmin(aniso_pair(txm, axm, tym, aym), aniso_pair(txm, axm, typ, ayp)));
    t = fmin(t, fmin(aniso_pair(txp, axp, tym, aym), aniso_pair(txp, axp, typ, ayp)));
    return t;
}

static int aniso_passable(const double* A, size_t plane, size_t q)
{
    return A[q] < ORC_INF || A[plane + q] < ORC_INF || A[2 * plane + q] < ORC_INF || A[3 * plane + q] < ORC_INF;
}

/* Heap-ordered march of the update from T(goal) = 0 (exact for an upwind update: a cell's value
 * only depends on neighbours with smaller values, which are final when it is popped).  T: nx*ny
 * doubles out, +inf where unreached.  Returns 0 if the goal is impassable (nothing seeded). */
int orc_aniso_march(const double* A, uint32_t nx, uint32_t ny, uint32_t gi, uint32_t gj, double* T)
{
    const size_t n = (size_t)nx * ny;
    for (size_t k = 0; k < n; ++k) T[k] = ORC_INF;
    const size_t g = (size_t)gj * nx + gi;
    if (gi >= nx || gj >= ny || !aniso_passable(A, n, g)) return 0;
    uint8_t* closed = (uint8_t*)calloc(n, 1);
    heap_t H;
    memset(&H, 0, sizeof(H));
    H.pos = (int64_t*)malloc(n * sizeof(int64_t));
    for (size_t k = 0; k < n; ++k) H.pos[k] = -1;
    T[g] = 0;
    hpush_or_decrease(&H, (uint32_t)g, 0.0);
    while (H.n)
    {
        const size_t k = hpop(&H);
        closed[k] = 1;
        const uint32_t i = (uint32_t)(k % nx), j = (uint32_t)(k / nx);
        const int has[4] = {i > 0, i + 1 < nx, j > 0, j + 1 < ny};
        const int64_t off[4] = {-1, 1, -(int64_t)nx, (int64_t)nx};
        for (int d = 0; d < 4; ++d)
        {
            if (!has[d]) continue;
            const size_t m = (size_t)((int64_t)k + off[d]);
            if (closed[m] || !aniso_passable(A, n, m)) continue;
            const double t = aniso_update(A, T, nx, ny, m);
            if (t < T[m])
            {
                T[m] = t;
                hpush_or_decrease(&H, (uint32_t)m, t);
            }
        }
    }
    free(H.h);
    free(H.pos);
    free(closed);
    return 1;
}

/* cells (other than the goal) whose update would lower T by more than rel_tol * T */
uint64_t orc_aniso_improvable(const double* A, const double* T, uint32_t nx, uint32_t ny, uint32_t gi,
                              uint32_t gj, double rel_tol)
{
    const size_t n = (size_t)nx * ny, g = (size_t)gj * nx + gi;
    uint64_t bad = 0;
    for (size_t q = 0; q < n; ++q)
    {
        if (q == g || !aniso_passable(A, n, q)) continue;
        const double t = aniso_update(A, T, nx, ny, q);
        if (t < T[q] - rel_tol * T[q]) bad++;
    }
    return bad;
}

/* node vector of the anisotropic descent (dymu_path.cu build_window<true>) at node (i, j) */
static void aniso_node_vector(const double* A, const double* T, uint32_t nx, uint32_t ny, uint32_t i, uint32_t j,
                              double* dnx, double* dny)
{
    const size_t plane = (size_t)nx * ny, q = (size_t)j * nx + i;
    const int64_t k = (int64_t)q;
    double dx = grad_axis(T, k, i > 0 ? k - 1 : -1, i + 1 < nx ? k + 1 : -1);
    double dy = grad_axis(T, k, j > 0 ? k - (int64_t)nx : -1, j + 1 < ny ? k + (int64_t)nx : -1);
    const double axm = A[q], axp = A[plane + q], aym = A[2 * plane + q], ayp = A[3 * plane + q];
    if (!(axm == ORC_INF && axp == ORC_INF && aym == ORC_INF && ayp == ORC_INF))
    {
        const double ax = dx > 0 ? axm : axp, ay = dy > 0 ? aym : ayp;
        dx = (dx == 0 || ax == ORC_INF) ? 0.0 : dx / (ax * ax);
        dy = (dy == 0 || ay == ORC_INF) ? 0.0 : dy / (ay * ay);
    }
    *dnx = *dny = 0;
    if (!(dx == 0 && dy == 0))
    {
        const double nrm = sqrt(dx * dx + dy * dy);
        *dnx = dx / nrm;
        *dny = dy / nrm;
    }
}

/* The walker of dymu_extract_global_path on the anisotropic node vectors.  out: 5 doubles per
 * waypoint {x, y, z, dCostX, dCostY}, the goal not appended; *status as DYMU_PATH_* (0 ok, 1 NaN,
 * 2 stalled, 3 capacity, 4 outside).  Returns the number of waypoints. */
uint32_t orc_aniso_path(const double* A, const double* T, const double* elev, uint32_t nx, uint32_t ny, double gres,
                        double x0, double y0, double tau, uint32_t goal_i, uint32_t goal_j, double* out, uint32_t cap,
                        int* status)
{
    const double sx = gres * (double)goal_i, sy = gres * (double)goal_j;
    const double c_step = gres * tau;
    const double lim_x = (double)(nx - 1), lim_y = (double)(ny - 1);
    const double far = 2.0 * gres, stall = 0.01 * tau * gres;
    uint32_t n = 0;
    double wx = x0, wy = y0, px = NAN, py = NAN;
    *status = 0;
    for (int first = 1;; first = 0)
    {
        const double gx = wx / gres, gy = wy / gres;
        const int outside = !(gx >= 0.0) || !(gy >= 0.0) || !(gx < lim_x) || !(gy < lim_y);
        if (first && outside) { *status = 4; break; }
        if (!first)
        {
            const double dp = sqrt((px - wx) * (px - wx) + (py - wy) * (py - wy));
            const double dg = sqrt((wx - sx) * (wx - sx) + (wy - sy) * (wy - sy));
            if (dp < stall) { *status = 2; break; }
            if (!(dg > far)) break;
            if (outside) { *status = 4; break; }
            if (n >= cap) { *status = 3; break; }
        }
        const uint32_t cx = (uint32_t)gx, cy = (uint32_t)gy;
        const double da = gx - trunc(gx), db = gy - trunc(gy);
        double vx[4], vy[4];  /* corners 00, 10, 01, 11 */
        aniso_node_vector(A, T, nx, ny, cx, cy, &vx[0], &vy[0]);
        aniso_node_vector(A, T, nx, ny, cx + 1, cy, &vx[1], &vy[1]);
        aniso_node_vector(A, T, nx, ny, cx, cy + 1, &vx[2], &vy[2]);
        aniso_node_vector(A, T, nx, ny, cx + 1, cy + 1, &vx[3], &vy[3]);
        const size_t q = (size_t)cy * nx + cx;
        const double dCx = interp(da, db, vx[0], vx[2], vx[1], vx[3]);
        const double dCy = interp(da, db, vy[0], vy[2], vy[1], vy[3]);
        const double z = interp(da, db, elev[q], elev[q + 1], elev[q + nx], elev[q + nx + 1]);
        const double nxt = wx - c_step * dCx, nyt = wy - c_step * dCy;
        if (first && (isnan(nxt) || isnan(nyt))) { *status = 1; break; }
        double* o = out + (size_t)5 * n;
        o[0] = wx; o[1] = wy; o[2] = z; o[3] = dCx; o[4] = dCy;
        n++;
        if (!first) { px = wx; py = wy; }  /* the first waypoint has no stall test */
        wx = nxt; wy = nyt;
    }
    return n;
}
