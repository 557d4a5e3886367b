"""Slope-anisotropic total-cost solve and descent (dymu_set_anisotropy) on the device, against the
isotropic solve (flat table), the plain-C restatement (oracle/dymu_oracle_aniso.c) and closed
forms."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TABLE = ([-20.0, -5.0, 0.0, 10.0, 25.0], [0.6, 0.8, 1.0, 1.8, 3.5])
FLAT = ([-90.0, 90.0], [1.0, 1.0])
DIRS = ("dircost_xm", "dircost_xp", "dircost_ym", "dircost_yp")
ERR_ARG, ERR_STATE = -2, -3


@pytest.fixture(scope="module")
def orc_aniso():
    """The plain-C restatement of the anisotropic model (built on first use)."""
    import oracle_aniso
    return oracle_aniso


def _mars(pkg, nx, ny, seed, table=None):
    syn = pkg.synthetic
    elev, terr = syn.mars_dem(ny, nx, seed=seed)
    lut, slopes, locs = syn.default_lut()
    dev = pkg.cuda_api.DeviceLayer(nx, ny, 1.0, 0.1)
    dev.compute_cost_map(lut, slopes, len(locs), elev, terr)
    if table is not None:
        dev.set_anisotropy(*table)
    ob = dev.download_plane_u8("obstacle")
    goal = syn.free_interior_cell_near(ob, int(nx * 0.8), int(ny * 0.7))
    start = syn.free_interior_cell_near(ob, int(nx * 0.15), int(ny * 0.2))
    return dev, elev, ob, goal, start


def _planes(dev):
    return np.stack([dev.download_plane(d) for d in DIRS])


def _rel(a, b):
    m = np.isfinite(b) & (b > 0)
    return float(np.max(np.abs(a[m] - b[m]) / b[m])) if m.any() else 0.0


def _same_path(a, b, tol=1e-3):
    (pa, sa), (pb, sb) = a, b
    assert sa == sb and len(pa) == len(pb)
    assert np.max(np.abs(pa[:, :2] - pb[:, :2])) <= tol


@pytest.mark.parametrize("n", [(257, 129), (1000, 1000)])
def test_flat_table_equals_isotropic(pkg, n):
    nx, ny = n
    iso, _, _, goal, start = _mars(pkg, nx, ny, seed=7)
    ani, _, _, _, _ = _mars(pkg, nx, ny, seed=7, table=FLAT)
    for dev in (iso, ani):
        assert dev.solve_total_cost([goal])["converged"]
    Ti, Ta = iso.download_total_cost(), ani.download_total_cost()
    assert np.array_equal(np.isinf(Ti), np.isinf(Ta))
    assert _rel(Ta, Ti) <= 1e-13
    _same_path(iso.extract_global_path(float(start[0]), float(start[1]), 0.4, *goal),
               ani.extract_global_path(float(start[0]), float(start[1]), 0.4, *goal))


@pytest.mark.parametrize("n", [(257, 129), (1000, 1000)])
def test_mars_against_oracle(pkg, orc_aniso, n):
    nx, ny = n
    dev, elev, ob, goal, start = _mars(pkg, nx, ny, seed=11, table=TABLE)
    A = _planes(dev)
    A_orc = orc_aniso.aniso_dircost(elev, dev.download_plane("ceff"), 1.0, *TABLE)
    assert np.array_equal(np.isinf(A), np.isinf(A_orc))
    assert _rel(A, A_orc) <= 1e-14
    st = dev.solve_total_cost([goal])
    assert st["converged"]
    T = dev.download_total_cost()
    T_orc = orc_aniso.aniso_march(A, goal)
    assert np.array_equal(np.isinf(T), np.isinf(T_orc))
    assert _rel(T, T_orc) <= 1e-9
    wps, status = dev.extract_global_path(float(start[0]), float(start[1]), 0.4, *goal)
    ref, ref_status = orc_aniso.aniso_path(A, T, elev, 1.0, start, 0.4, goal)
    _same_path((wps, status), (ref, ref_status))
    # the direction-dependent map differs from the isotropic one
    iso, _, _, _, _ = _mars(pkg, nx, ny, seed=11)
    iso.solve_total_cost([goal])
    assert _rel(T, iso.download_total_cost()) > 1e-3


def test_corridor_is_exact_and_asymmetric(pkg):
    n, c, slope = 64, 0.7, 10.0
    dev = pkg.cuda_api.DeviceLayer(n, 3, 1.0, 0.1)
    cost = np.zeros((3, n))
    cost[1, :] = c  # C_eff = 1 * cost * (2 + hazard 0 - trafficability 1) on free cells
    dev.set_cost_map(cost)
    assert np.all(dev.download_plane("ceff")[1] == c)
    elev = np.tile(np.arange(n, dtype=np.float64) * math.tan(math.radians(slope)), (3, 1))
    dev.upload_plane("elevation", elev)
    table = ([-20.0, 0.0, 20.0], [0.5, 1.0, 3.0])
    dev.set_anisotropy(*table)
    th = math.degrees(math.atan(math.tan(math.radians(slope))))
    up, down = c * np.interp(th, *table), c * np.interp(-th, *table)
    goal = 30
    dev.solve_total_cost([(goal, 1)])
    T = dev.download_total_cost()[1]
    expect = np.zeros(n)
    for i in range(goal + 1, n):
        expect[i] = expect[i - 1] + down
    for i in range(goal - 1, -1, -1):
        expect[i] = expect[i + 1] + up
    assert _rel(T, expect) <= 1e-12
    # swapping goal and start: the climb costs what the table says
    d = 12
    dev.solve_total_cost([(goal - d, 1)])
    T_up_goal = dev.download_total_cost()[1][goal]
    assert T_up_goal / T[goal - d] == pytest.approx(down / up, rel=1e-12)


def test_plan4096_fixed_point_delivery_and_descent(pkg):
    n = 4096
    dev, _, ob, _, _ = _mars(pkg, n, n, seed=20261018, table=TABLE)
    goal = pkg.synthetic.free_interior_cell_near(ob, n // 2, n // 2)
    import torch
    pinned = torch.empty((n, n), dtype=torch.float64, pin_memory=True).numpy()
    assert dev.set_total_cost_export(pinned, pkg.cuda_api.XFORM_INF_TO_MINUS1)
    st = dev.solve_total_cost([goal])
    dev.synchronize()
    assert st["converged"] and st["tiles_delivered_early"] > 0
    T = dev.download_total_cost()
    assert np.array_equal(pinned, np.where(np.isinf(T), -1.0, T))
    dev.set_total_cost_export(None)
    A = _planes(dev)
    # the update on whole planes (expression order of k_fim's relax_aniso) improves no cell
    P = np.pad(T, 1, constant_values=np.inf)
    nb = (P[1:-1, :-2], P[1:-1, 2:], P[:-2, 1:-1], P[2:, 1:-1])
    del P
    with np.errstate(invalid="ignore", over="ignore"):
        best = np.minimum(np.minimum(nb[0] + A[0], nb[1] + A[1]), np.minimum(nb[2] + A[2], nb[3] + A[3]))
        for h in (0, 1):
            for v in (2, 3):
                Th, ah, Tv, av = nb[h], A[h], nb[v], A[v]
                d = Th - Tv
                s = ah * ah + av * av
                ok = (d > -ah) & (d < av) & (s < np.inf)
                t = ((av * av * Th + ah * ah * Tv) + (ah * av) * np.sqrt(np.where(ok, s - d * d, 1.0))) / s
                best = np.minimum(best, np.where(ok, t, np.inf))
    target = np.isfinite(A).any(axis=0)
    target[goal[1], goal[0]] = False
    assert not (best[target] < T[target] * (1 - 1e-14)).any()
    del best, A
    start = pkg.synthetic.free_interior_cell_near(ob, n // 16, n // 16)
    wps, status = dev.extract_global_path(float(start[0]), float(start[1]), 0.4, goal[0], goal[1])
    assert status == 0 and len(wps) > n // 4
    ij = np.rint(wps[:, :2]).astype(np.int64)
    t_along = T[ij[:, 1], ij[:, 0]]
    assert np.isfinite(t_along).all() and (np.diff(t_along[::25]) < 0).all()
    assert np.hypot(wps[-1, 0] - goal[0], wps[-1, 1] - goal[1]) <= 2.0 + 0.4


def test_eight_goals_in_one_launch(pkg):
    nx, ny = 513, 385
    dev, _, ob, _, _ = _mars(pkg, nx, ny, seed=3, table=TABLE)
    syn = pkg.synthetic
    goals = [syn.free_interior_cell_near(ob, 40 + 55 * k, 30 + 40 * k) for k in range(8)]
    dev.reserve_slots(8)
    assert dev.solve_total_cost(goals)["converged"]
    batch = [dev.download_total_cost(slot=k) for k in range(8)]
    one, _, _, _, _ = _mars(pkg, nx, ny, seed=3, table=TABLE)
    for k, g in enumerate(goals):
        one.solve_total_cost([g])
        T = one.download_total_cost()
        assert np.array_equal(np.isinf(T), np.isinf(batch[k])) and _rel(batch[k], T) <= 1e-13


def test_switching_off_restores_isotropic(pkg):
    nx, ny = 300, 200
    never, _, _, goal, start = _mars(pkg, nx, ny, seed=5)
    was, _, _, _, _ = _mars(pkg, nx, ny, seed=5, table=TABLE)
    was.solve_total_cost([goal])
    was.set_anisotropy([], [])
    with pytest.raises(pkg.cuda_api.DymuError):
        was.download_plane("dircost_xm")
    for dev in (never, was):
        dev.solve_total_cost([goal])
    assert _rel(was.download_total_cost(), never.download_total_cost()) <= 1e-13
    _same_path(never.extract_global_path(float(start[0]), float(start[1]), 0.4, *goal),
               was.extract_global_path(float(start[0]), float(start[1]), 0.4, *goal))


def test_entry_points(pkg, orc_aniso):
    nx, ny = 320, 256
    dev, elev, ob, goal, _ = _mars(pkg, nx, ny, seed=13, table=TABLE)
    err = pkg.cuda_api.DymuError
    for bad in (([0.0], [1.0]), ([0.0, 0.0], [1.0, 1.0]), ([1.0, 0.0], [1.0, 1.0]), ([0.0, 1.0], [1.0, 0.0]),
                ([0.0, float("nan")], [1.0, 1.0]), ([0.0, 1.0], [1.0, float("inf")])):
        with pytest.raises(err) as e:
            dev.set_anisotropy(*bad)
        assert e.value.code == ERR_ARG
    with pytest.raises(err) as e:
        dev.upload_plane("dircost_yp", np.zeros((ny, nx)))
    assert e.value.code == ERR_ARG
    with pytest.raises(err) as e:
        dev.solve_start(goal, 4)
    assert e.value.code == ERR_STATE
    with pytest.raises(err) as e:
        dev.solve_advance([(0, 32)], 0.0, 4)
    assert e.value.code == ERR_STATE
    dev.solve_total_cost([goal])
    T0 = dev.download_total_cost()
    st, inv = dev.solve_incremental(goal)
    assert inv is None and st["converged"]
    # a cost-map change after enabling reaches the directional costs and the solve
    cost = dev.download_plane("cost")
    cost[ny // 3: ny // 3 + 20, nx // 4: nx // 2] *= 3.0
    dev.upload_plane("cost", cost)
    st, inv = dev.solve_incremental(goal)
    assert inv is None
    T1 = dev.download_total_cost()
    A = _planes(dev)
    assert _rel(A, orc_aniso.aniso_dircost(elev, dev.download_plane("ceff"), 1.0, *TABLE)) <= 1e-14
    T_orc = orc_aniso.aniso_march(A, goal)
    assert np.array_equal(np.isinf(T1), np.isinf(T_orc)) and _rel(T1, T_orc) <= 1e-9
    assert _rel(T1, T0) > 1e-6
    # and so does a new elevation
    elev2 = elev * 1.5
    dev.upload_plane("elevation", elev2)
    dev.solve_total_cost([goal])
    A2 = _planes(dev)
    assert _rel(A2, orc_aniso.aniso_dircost(elev2, dev.download_plane("ceff"), 1.0, *TABLE)) <= 1e-14
    # the streamed plan uploads first and then solves in full
    cost_host = np.ascontiguousarray(cost)
    dev.plan_streamed(cost_host, goal)
    T2 = dev.download_total_cost()
    dev.set_cost_map(cost_host)
    dev.solve_total_cost([goal])
    assert np.array_equal(np.isinf(T2), np.isinf(dev.download_total_cost()))
    assert _rel(T2, dev.download_total_cost()) <= 1e-13
    # domain decomposition is isotropic only
    with pytest.raises(err) as e:
        pkg.cuda_api.dd_solve([dev], [0, ny], goal)
    assert e.value.code == ERR_STATE


def test_planner_class(pkg):
    nx, ny = 257, 193
    syn = pkg.synthetic
    elev, terr = syn.mars_dem(ny, nx, seed=17)
    lut, slopes, locs = syn.default_lut()
    p = pkg.DyMuPathPlanner(1.0, 1.5, 2.0, pkg.planner_api.SWEEPING)
    assert not p.setSlopeAnisotropy(*TABLE)  # before initGlobalLayer
    assert p.initGlobalLayer(1.0, 0.1, nx, ny)
    assert p.computeCostMap(lut, slopes, locs, elev, terr)
    assert not p.setSlopeAnisotropy([0.0, 0.0], [1.0, 1.0])
    assert p.setSlopeAnisotropy(*TABLE)
    ob = p.node_field(4)
    gi, gj = syn.free_interior_cell_near(ob, 200, 150)
    si, sj = syn.free_interior_cell_near(ob, 30, 30)
    assert p.setGoal(gi, gj) and p.computeEntireTotalCostMap()
    M = p.getTotalCostMatrix()
    path = p.getPath(si, sj)
    dev, _, _, _, _ = _mars(pkg, nx, ny, seed=17, table=TABLE)
    dev.solve_total_cost([(gi, gj)])
    T = dev.download_total_cost()
    assert np.array_equal(M < 0, np.isinf(T)) and _rel(M, T) <= 1e-13
    wps, status = dev.extract_global_path(float(si), float(sj), 0.4, gi, gj)
    assert status == 0 and len(path) == len(wps) + 1
    assert np.max(np.abs(path[:-1, :2] - wps[:, :2])) <= 1e-3
    # switching off through the class gives the isotropic plane again
    assert p.setSlopeAnisotropy([], []) and p.computeEntireTotalCostMap()
    iso, _, _, _, _ = _mars(pkg, nx, ny, seed=17)
    iso.solve_total_cost([(gi, gj)])
    Ti = iso.download_total_cost()
    assert _rel(p.getTotalCostMatrix(), Ti) <= 1e-13
