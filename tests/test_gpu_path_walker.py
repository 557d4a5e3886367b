"""Global path extraction against a scalar restatement of the reference walk.

`walk` restates gradientNode, interpolate, computeNextGlobalWaypoint and the computeGlobalPath
loop (src/DyMu_GlobalPathPlanning.cpp:615-784) on the total-cost and elevation planes
downloaded from the device.  Python floats are IEEE doubles, every operation is rounded on
its own (no fused multiply-add) and math.sqrt and / are correctly rounded, so the device walk
must reproduce it bit for bit: waypoints, count and status.  The cases cover window changes
over a long path, grid edges and corners, a U-turn around a wall, unreachable and obstacle
starts, stalls, a small capacity, several step sizes, a global resolution of 0.5 and the
batched call."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

OK, NAN, STALLED, CAPACITY, OUTSIDE = 0, 1, 2, 3, 4
INF = float("inf")


def _grad_axis(f, has_lo, flo, has_hi, fhi):
    if (not has_lo and not has_hi) or (has_lo and has_hi and flo == INF and fhi == INF):
        return 0.0
    if not has_lo or flo == INF:
        if not has_hi:
            return 0.0
        return fhi - f
    if not has_hi or fhi == INF:
        return f - flo
    return (fhi - flo) * 0.5


def _gradient(T, i, j):
    """gradientNode: normalised gradient of the total cost at node (i, j) = (column, row)."""
    ny, nx = T.shape
    f = float(T[j, i])
    hl, hr, hd, hu = i > 0, i + 1 < nx, j > 0, j + 1 < ny
    fl = float(T[j, i - 1]) if hl else 0.0
    fr = float(T[j, i + 1]) if hr else 0.0
    fd = float(T[j - 1, i]) if hd else 0.0
    fu = float(T[j + 1, i]) if hu else 0.0
    dx = _grad_axis(f, hl, fl, hr, fr)
    dy = _grad_axis(f, hd, fd, hu, fu)
    if dx == 0 and dy == 0:
        return 0.0, 0.0
    n = math.sqrt(dx * dx + dy * dy)
    return dx / n, dy / n


def _interp(a, b, g00, g01, g10, g11):
    return g00 + (g10 - g00) * a + (g01 - g00) * b + (g11 + g00 - g10 - g01) * a * b


def _next(T, E, gres, tau, wx, wy):
    """computeNextGlobalWaypoint; None when the cell leaves the grid."""
    ny, nx = T.shape
    gx, gy = wx / gres, wy / gres
    if not (gx >= 0.0) or not (gy >= 0.0) or not (gx < float(nx - 1)) or not (gy < float(ny - 1)):
        return None
    cx, cy = int(gx), int(gy)
    da, db = gx - float(cx), gy - float(cy)
    g00, g10 = _gradient(T, cx, cy), _gradient(T, cx + 1, cy)
    g01, g11 = _gradient(T, cx, cy + 1), _gradient(T, cx + 1, cy + 1)
    dcx = _interp(da, db, g00[0], g01[0], g10[0], g11[0])
    dcy = _interp(da, db, g00[1], g01[1], g10[1], g11[1])
    e00, e10 = float(E[cy, cx]), float(E[cy, cx + 1])
    e01, e11 = float(E[cy + 1, cx]), float(E[cy + 1, cx + 1])
    z = _interp(da, db, e00, e10, e01, e11)  # the reference's swapped corner order
    return z, dcx, dcy, wx - gres * tau * dcx, wy - gres * tau * dcy


def walk(T, E, gres, tau, x0, y0, goal, cap):
    """computeGlobalPath with the device's statuses: (waypoints (n, 5), status)."""
    out = []
    r = _next(T, E, gres, tau, x0, y0)
    if r is None:
        return np.zeros((0, 5)), OUTSIDE
    z, dcx, dcy, nx_, ny_ = r
    if math.isnan(nx_) or math.isnan(ny_):
        return np.zeros((0, 5)), NAN
    out.append((x0, y0, z, dcx, dcy))
    wx, wy = nx_, ny_
    sx, sy = gres * float(goal[0]), gres * float(goal[1])
    status = OK
    while math.sqrt((wx - sx) * (wx - sx) + (wy - sy) * (wy - sy)) > 2.0 * gres:
        r = _next(T, E, gres, tau, wx, wy)
        if r is None:
            status = OUTSIDE
            break
        if len(out) >= cap:
            status = CAPACITY
            break
        z, dcx, dcy, nx_, ny_ = r
        out.append((wx, wy, z, dcx, dcy))
        if math.sqrt((wx - nx_) * (wx - nx_) + (wy - ny_) * (wy - ny_)) < 0.01 * tau * gres:
            status = STALLED
            break
        wx, wy = nx_, ny_
    return np.array(out, dtype=np.float64).reshape(-1, 5), status


def _same_bits(a, b):
    a, b = np.ascontiguousarray(a, np.float64), np.ascontiguousarray(b, np.float64)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint64), b[~nb].view(np.uint64)))


def _check(dev, gres, tau, start, goal, cap=1 << 18, planes=None):
    T, E = planes if planes is not None else (dev.download_total_cost(), dev.download_plane("elevation"))
    want, want_status = walk(T, E, gres, tau, float(start[0]), float(start[1]), goal, cap)
    got, status = dev.extract_global_path(float(start[0]), float(start[1]), tau, goal[0], goal[1], cap=cap)
    assert status == want_status, (start, goal, tau, status, want_status)
    assert len(got) == len(want), (start, goal, tau, len(got), len(want))
    assert _same_bits(got, want), (start, goal, tau)
    return len(got), status


def _mars(pkg, n, gres=1.0, seed=7):
    syn = pkg.synthetic
    elev, terr = syn.mars_dem(n, n, seed=seed)
    lut, slopes, locs = syn.default_lut()
    dev = pkg.cuda_api.DeviceLayer(n, n, gres, 0.1)
    dev.compute_cost_map(lut, slopes, len(locs), elev, terr)
    return dev, dev.download_plane_u8("obstacle")


def _wall_map(pkg, n=384):
    """Uniform cost with a wall from the bottom edge to 3/4 of the height at x = n/2, and a
    closed box (unreachable inside) in the top-left corner."""
    cost = np.ones((n, n))
    cost[: 3 * n // 4, n // 2] = 0.0
    cost[n - 60: n - 20, 20] = cost[n - 60: n - 20, 60] = 0.0
    cost[n - 60, 20:61] = cost[n - 20, 20:61] = 0.0
    dev = pkg.cuda_api.DeviceLayer(n, n)
    dev.set_cost_map(cost)
    y, x = np.mgrid[0:n, 0:n]
    dev.upload_plane("elevation", np.sin(x * 0.05) * np.cos(y * 0.03) * 10.0)
    return dev


def test_bench_map_long_path(pkg):
    """The 4096^2 benchmark map, goal and start: a path of thousands of waypoints crossing
    many windows."""
    n = 4096
    syn = pkg.synthetic
    elev, terr = syn.mars_dem(n, n, seed=20261018)
    lut, slopes, locs = syn.default_lut()
    dev = pkg.cuda_api.DeviceLayer(n, n, 1.0, 0.1)
    dev.compute_cost_map(lut, slopes, len(locs), elev, terr)
    ob = dev.download_plane_u8("obstacle")
    goal = syn.free_interior_cell_near(ob, n // 2, n // 2)
    start = syn.free_interior_cell_near(ob, n // 8, n // 8)
    dev.solve_total_cost([goal])
    count, status = _check(dev, 1.0, 0.4, start, goal)
    assert status == OK and count > 3000
    # capacity: the walk stops with exactly `cap` waypoints
    planes = (dev.download_total_cost(), dev.download_plane("elevation"))
    assert _check(dev, 1.0, 0.4, start, goal, cap=37, planes=planes) == (37, CAPACITY)
    dev.close()


@pytest.mark.parametrize("tau", [0.1, 0.4, 1.5])
def test_edges_and_corners(pkg, tau):
    """Starts next to every grid edge and corner, and goals in the corners, so windows are
    clipped by the grid on every side.  The map's border cells are obstacles: starts on them
    end at once (NaN step), starts on or past the last row or column leave the grid."""
    n = 256
    dev, ob = _mars(pkg, n)
    syn = pkg.synthetic
    e = n - 1
    near = [(0, 0), (e, 0), (0, e), (e, e), (0, n // 2), (e, n // 3), (n // 2, 0), (n // 3, e)]
    starts = [tuple(float(v) + 0.25 for v in syn.free_interior_cell_near(ob, *c)) for c in near]
    starts += [(0.0, 0.0), (e - 0.5, e - 0.5), (e, 5.0), (-0.5, 5.0)]
    goals = [syn.free_interior_cell_near(ob, n // 2, n // 2), syn.free_interior_cell_near(ob, 3, 3),
             syn.free_interior_cell_near(ob, e - 3, 3), syn.free_interior_cell_near(ob, e - 3, e - 3)]
    seen = set()
    for goal in goals:
        dev.solve_total_cost([goal])
        planes = (dev.download_total_cost(), dev.download_plane("elevation"))
        for s in starts:
            seen.add(_check(dev, 1.0, tau, s, goal, planes=planes)[1])
    assert OUTSIDE in seen and OK in seen
    dev.close()


def test_wall_turn_unreachable_and_obstacle_starts(pkg):
    """A U-turn around a wall (the window ahead of the walker is the wrong one), starts in an
    unreachable box (a stall: zero gradient) and on an obstacle."""
    n = 384
    dev = _wall_map(pkg, n)
    goal = (3 * n // 4, n // 4)
    dev.solve_total_cost([goal])
    planes = (dev.download_total_cost(), dev.download_plane("elevation"))
    seen = {}
    for tau in (0.1, 0.4, 1.5):
        for s in [(n / 4, n / 4), (n / 2 - 2.5, 10.0), (40.0, n - 40.0), (n / 2, 100.0), (20.0, n - 40.0),
                  (n / 2 - 0.5, n / 2)]:
            cnt, st = _check(dev, 1.0, tau, s, goal, planes=planes)
            seen.setdefault(st, cnt)
    assert seen.get(OK, 0) > 300  # the U-turn path
    assert STALLED in seen
    dev.close()


@pytest.mark.parametrize("tau", [0.1, 0.4, 1.5])
def test_global_resolution_half(pkg, tau):
    n = 320
    dev, ob = _mars(pkg, n, gres=0.5, seed=11)
    syn = pkg.synthetic
    goal = syn.free_interior_cell_near(ob, 2 * n // 3, n // 3)
    dev.solve_total_cost([goal])
    planes = (dev.download_total_cost(), dev.download_plane("elevation"))
    for c in [(20, 20), (n - 10, n - 10), (5, n - 5), (n // 2, n - 2)]:
        s = syn.free_interior_cell_near(ob, *c)
        cnt, st = _check(dev, 0.5, tau, (0.5 * s[0], 0.5 * s[1]), goal, planes=planes)
        assert st == OK and cnt > 10
    dev.close()


def test_batch_matches_single_calls(pkg):
    n = 512
    dev, ob = _mars(pkg, n, seed=3)
    syn = pkg.synthetic
    rng = np.random.default_rng(5)
    q = 12
    goals = [syn.free_interior_cell_near(ob, int(rng.uniform(0.05, 0.95) * n), int(rng.uniform(0.05, 0.95) * n))
             for _ in range(q)]
    starts = [[float(v) for v in syn.free_interior_cell_near(ob, int(rng.uniform(0.05, 0.95) * n),
                                                             int(rng.uniform(0.05, 0.95) * n))] for _ in range(q)]
    starts[3] = [-1.0, 4.0]
    dev.reserve_slots(q)
    dev.solve_total_cost(goals)
    paths, status = dev.extract_global_path_batch(list(range(q)), starts, 0.4, goals, cap=1 << 14)
    E = dev.download_plane("elevation")
    for k in range(q):
        single, st = dev.extract_global_path(starts[k][0], starts[k][1], 0.4, goals[k][0], goals[k][1], slot=k,
                                             cap=1 << 14)
        assert status[k] == st and _same_bits(paths[k], single), k
        want, want_st = walk(dev.download_total_cost(slot=k), E, 1.0, 0.4, starts[k][0], starts[k][1], goals[k],
                             1 << 14)
        assert st == want_st and _same_bits(single, want), k
    assert status[3] == OUTSIDE and sum(s == OK for s in status) >= q // 2
    dev.close()
