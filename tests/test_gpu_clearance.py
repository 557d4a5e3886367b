"""Obstacle clearance (dymu_set_obstacle_clearance) on the device: the clearance plane and C_eff against
the numpy model (tests/clearance_model.py), the solve against the reference port run on the transformed
cost map, path clearance, the incremental re-solve, slope anisotropy, the other entry points and the
planner class."""
import numpy as np
import pytest

import clearance_model as cm
import scenarios as sc

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_STATE = -2, -3
RMP = (2.0, 6.0, 4.0)  # radius, margin (metres), penalty
TABLE = ([-20.0, -5.0, 0.0, 10.0, 25.0], [0.6, 0.8, 1.0, 1.8, 3.5])
DIRS = ("dircost_xm", "dircost_xp", "dircost_ym", "dircost_yp")


def _mars(pkg, nx, ny, seed, clear=RMP):
    syn = pkg.synthetic
    elev, terr = syn.mars_dem(ny, nx, seed=seed)
    lut, slopes, locs = syn.default_lut()
    dev = pkg.cuda_api.DeviceLayer(nx, ny, 1.0, 0.1)
    dev.compute_cost_map(lut, slopes, len(locs), elev, terr)
    if clear is not None:
        dev.set_obstacle_clearance(*clear)
    return dev, elev


def _model(dev, radius, margin, penalty, g=1.0):
    ob = dev.download_plane_u8("obstacle")
    d = cm.clearance(ob, radius, margin, g)
    c = cm.plain_ceff(dev.download_plane("cost"), dev.download_plane("hazard_density"),
                      dev.download_plane("trafficability"), ob, g)
    return d, cm.ceff(c, d, radius, margin, penalty)


def _check_model(dev, rmp, g=1.0):
    d, C = _model(dev, *rmp, g=g)
    assert np.array_equal(dev.download_plane("clearance"), d)
    assert np.array_equal(dev.download_plane("ceff"), C)
    return d, C


def _free_goal_start(pkg, blocked, nx, ny):
    syn = pkg.synthetic
    return (syn.free_interior_cell_near(blocked, int(nx * 0.8), int(ny * 0.7)),
            syn.free_interior_cell_near(blocked, int(nx * 0.15), int(ny * 0.2)))


def _rel(a, b):
    m = np.isfinite(b) & (b > 0)
    return float(np.max(np.abs(a[m] - b[m]) / b[m])) if m.any() else 0.0


def _same_T(a, b, tol):
    assert np.array_equal(np.isinf(a), np.isinf(b))
    assert _rel(a, b) <= tol


# ---- 1. planes against the model ---------------------------------------------------------------
@pytest.mark.parametrize("n", [(257, 129), (1000, 1000)])
@pytest.mark.parametrize("rmp", [RMP, (0.0, 3.0, 2.0), (3.0, 0.0, 0.0), (60.0, 68.5, 1.0)])
def test_planes_equal_model_on_mars(pkg, n, rmp):
    dev, _ = _mars(pkg, *n, seed=11, clear=rmp)
    d, C = _check_model(dev, rmp)
    assert (np.isfinite(d) & (d > 0)).any()


def test_obstacles_on_the_border(pkg):
    nx, ny, g = 203, 77, 0.5
    rng = np.random.default_rng(3)
    cost = rng.uniform(0.2, 2.0, (ny, nx))
    cost[0, 5:9] = cost[-1, 100] = cost[30, 0] = cost[40:44, -1] = 0.0
    cost[rng.integers(0, ny, 40), rng.integers(0, nx, 40)] = 0.0
    dev = pkg.cuda_api.DeviceLayer(nx, ny, g, 0.1)
    dev.set_cost_map(cost)
    rmp = (1.0, 1.75, 3.0)
    dev.set_obstacle_clearance(*rmp)
    _check_model(dev, rmp, g=g)


# ---- 2. switching off ---------------------------------------------------------------------------
def test_off_is_bit_identical_to_never_enabled(pkg):
    nx, ny = 300, 200
    a, _ = _mars(pkg, nx, ny, seed=3)
    b, _ = _mars(pkg, nx, ny, seed=3, clear=None)
    goal, start = _free_goal_start(pkg, a.download_plane_u8("obstacle"), nx, ny)
    a.solve_total_cost([goal])
    a.set_obstacle_clearance(0.0, 0.0, 0.0)
    with pytest.raises(pkg.cuda_api.DymuError) as e:
        a.download_plane("clearance")
    assert e.value.code == ERR_ARG
    for dev in (a, b):
        assert dev.solve_total_cost([goal])["converged"]
    assert np.array_equal(a.download_plane("ceff"), b.download_plane("ceff"))
    # the solver's update order varies from run to run, and with it the last bits of the total cost
    # (bench.py --dump-outputs): two solves of one context differ as much
    _same_T(a.download_total_cost(), b.download_total_cost(), 1e-13)
    pa, sa = a.extract_global_path(float(start[0]), float(start[1]), 0.4, *goal)
    pb, sb = b.extract_global_path(float(start[0]), float(start[1]), 0.4, *goal)
    assert sa == sb and pa.shape == pb.shape and np.max(np.abs(pa[:, :2] - pb[:, :2])) <= 1e-9


def test_plane_is_read_only(pkg):
    dev, _ = _mars(pkg, 100, 90, seed=4)
    dev.download_plane("clearance")
    for call in (lambda: dev.write_rect("clearance", 0, 0, np.zeros((2, 2))),
                 lambda: dev.upload_plane("clearance", np.zeros((90, 100))),
                 lambda: dev.plane_device_ptr("clearance")):
        with pytest.raises(pkg.cuda_api.DymuError) as e:
            call()
        assert e.value.code == ERR_ARG


# ---- 3. parity with the reference port on the transformed cost map ----------------------------
@pytest.mark.parametrize("n,solves", [(1000, (False, True)), (2048, (True,))])
def test_parity_with_port_on_transformed_map(pkg, oracle_mod, n, solves):
    syn = pkg.synthetic
    radius, margin, penalty = RMP
    cost = syn.smooth_cost_map(n, n, seed=21)
    d = cm.clearance(cost <= 0, radius, margin, 1.0)
    band = (d > radius) & (d < radius + margin)
    cost_t = np.where(d <= radius, 0.0, np.where(band, cost * cm.factor(d, radius, margin, penalty), cost))
    (gi, gj), (si, sj) = _free_goal_start(pkg, (cost_t <= 0).astype(np.float64), n, n)
    dut = pkg.DyMuPathPlanner(1.0, 1.5, 2.0, pkg.planner_api.SWEEPING)
    assert dut.initGlobalLayer(1.0, 0.1, n, n)
    assert dut.setCostMap(cost) and dut.setObstacleClearance(radius, margin, penalty)
    assert dut.setGoal(gi, gj) and dut.computeEntireTotalCostMap()
    T, path = dut.getTotalCostMatrix(), dut.getPath(si, sj)
    for heap in solves:
        chk = oracle_mod.Port(1.0, 1.5, 2.0, oracle_mod.SWEEPING)
        assert chk.initGlobalLayer(1.0, 0.1, n, n)
        assert chk.setCostMap(cost_t) and chk.setGoal(gi, gj)
        assert chk.computeEntireTotalCostMap(heap=heap)
        Tr = chk.getTotalCostMatrix()
        assert np.array_equal(T < 0, Tr < 0)
        fin = Tr > 0
        assert float(np.max(np.abs(T[fin] - Tr[fin]) / Tr[fin])) <= 1e-9
        pr = chk.getPath(si, sj)
        assert path.shape == pr.shape and float(np.max(np.abs(path[:, :2] - pr[:, :2]))) <= 1e-3
        chk.close()


# ---- 4. the path keeps its distance ------------------------------------------------------------
def test_path_keeps_clear_of_the_rock(pkg):
    nx, ny = 60, 25
    cost = np.ones((ny, nx))
    cost[0, :] = cost[-1, :] = 0.0  # corridor walls
    rock = (30, 12)
    cost[rock[1], rock[0]] = 0.0
    obst = np.argwhere(cost <= 0)[:, ::-1].astype(np.float64)  # (i, j) of the obstacle cells
    # one row off the rock's row: on the axis of the symmetric corridor the descent would stall on the
    # ridge between the two ways round
    start, goal = (4, 11), (56, 11)

    def min_dist(dev):
        wps, status = dev.extract_global_path(float(start[0]), float(start[1]), 0.4, *goal)
        assert status == 0 and len(wps) > 10
        xy = wps[:, :2]
        return float(np.min(np.hypot(xy[:, None, 0] - obst[None, :, 0], xy[:, None, 1] - obst[None, :, 1])))

    dev = pkg.cuda_api.DeviceLayer(nx, ny, 1.0, 0.1)
    dev.set_cost_map(cost)
    dev.solve_total_cost([goal])
    assert min_dist(dev) < 2.0  # the point planner brushes the rock
    radius = 3.0
    dev.set_obstacle_clearance(radius, 2.0, 2.0)
    dev.solve_total_cost([goal])
    assert min_dist(dev) >= radius - np.sqrt(2) / 2


# ---- 5. incremental re-solve ------------------------------------------------------------------
def test_incremental_hazard_patch_and_new_obstacle(pkg):
    n = 1000
    dev, elev = _mars(pkg, n, n, seed=5)
    twin, _ = _mars(pkg, n, n, seed=5, clear=None)  # same calls without clearance
    goal, _ = _free_goal_start(pkg, dev.download_plane_u8("obstacle"), n, n)
    for d in (dev, twin):
        assert d.solve_total_cost([goal])["converged"]
    # the local layer's feedback: hazard up, trafficability down in a patch the wave crossed
    i0, j0, w = 400, 450, 40
    haz = dev.read_rect("hazard_density", i0, j0, w, w)
    tra = dev.read_rect("trafficability", i0, j0, w, w)
    launches = []
    for d in (dev, twin):
        d.write_rect("hazard_density", i0, j0, np.minimum(haz + 0.5, 1.0))
        d.write_rect("trafficability", i0, j0, np.maximum(tra - 0.3, 0.0))
        n0 = d.launches
        st, inv = d.solve_incremental(goal)
        launches.append(d.launches - n0)
        assert st["converged"] and inv is not None and 0 < inv < n * n // 4
    # the same kernels ran as without clearance: the distance transform did not
    assert launches[0] == launches[1]
    T_inc = dev.download_total_cost()
    _check_model(dev, RMP)
    dev.solve_total_cost([goal])
    _same_T(T_inc, dev.download_total_cost(), 1e-12)
    # a C_eff refresh after a hazard change is one pass on the resident clearance plane ...
    dev.write_rect("hazard_density", i0, j0, haz)
    n0 = dev.launches
    dev.download_plane("ceff")
    assert dev.launches - n0 == 1
    dev.solve_total_cost([goal])
    # ... an obstacle change rebuilds the plane (both passes), and the re-solve equals a fresh context
    cost = dev.download_plane("cost")
    cost[480:484, 700:703] = 0.0
    dev.set_cost_map(cost)
    st, inv = dev.solve_incremental(goal)
    assert st["converged"]
    T_inc = dev.download_total_cost()
    fresh, _ = _mars(pkg, n, n, seed=5, clear=None)
    fresh.write_rect("hazard_density", 0, 0, dev.download_plane("hazard_density"))
    fresh.write_rect("trafficability", 0, 0, dev.download_plane("trafficability"))
    fresh.set_cost_map(cost)
    fresh.set_obstacle_clearance(*RMP)
    fresh.solve_total_cost([goal])
    assert np.array_equal(fresh.download_plane("clearance"), dev.download_plane("clearance"))
    assert np.array_equal(fresh.download_plane("ceff"), dev.download_plane("ceff"))
    _same_T(T_inc, fresh.download_total_cost(), 1e-12)
    n0 = dev.launches
    dev.set_cost_map(cost)
    dev.download_plane("ceff")
    assert dev.launches - n0 == 3  # k_set_cost_map, column pass, fused row pass


# ---- 6. with slope anisotropy ------------------------------------------------------------------
def test_with_anisotropy(pkg):
    import oracle_aniso
    nx, ny = 257, 129
    dev, elev = _mars(pkg, nx, ny, seed=11)
    dev.set_anisotropy(*TABLE)
    _, C = _check_model(dev, RMP)
    A = np.stack([dev.download_plane(k) for k in DIRS])
    A_orc = oracle_aniso.aniso_dircost(elev, C, 1.0, *TABLE)
    assert np.array_equal(np.isinf(A), np.isinf(A_orc))
    assert _rel(A, A_orc) <= 1e-14
    goal, _ = _free_goal_start(pkg, dev.download_plane_u8("obstacle"), nx, ny)
    assert dev.solve_total_cost([goal])["converged"]
    T = dev.download_total_cost()
    T_orc = oracle_aniso.aniso_march(A, goal)
    _same_T(T, T_orc, 1e-9)


# ---- 7. other entry points --------------------------------------------------------------------
def test_eight_goals_in_one_launch(pkg):
    n = 300
    dev, _ = _mars(pkg, n, n, seed=8)
    ob = dev.download_plane_u8("obstacle")
    d = dev.download_plane("clearance")
    rng = np.random.default_rng(2)
    goals = []
    while len(goals) < 8:
        i, j = (int(v) for v in rng.integers(5, n - 5, 2))
        if not ob[j, i] and d[j, i] > RMP[0]:
            goals.append((i, j))
    dev.reserve_slots(8)
    dev.solve_total_cost(goals)
    multi = [dev.download_total_cost(slot=q) for q in range(8)]
    for q, g in enumerate(goals):
        dev.solve_total_cost([g])
        _same_T(multi[q], dev.download_total_cost(), 1e-13)


def test_batch_solve_on_two_contexts(pkg):
    n = 300
    layers = [_mars(pkg, n, n, seed=9)[0] for _ in range(2)]
    ob = layers[0].download_plane_u8("obstacle")
    d = layers[0].download_plane("clearance")
    blocked = ob.astype(bool) | (d <= RMP[0])
    goals = [pkg.synthetic.free_interior_cell_near(blocked, ci, cj)
             for ci, cj in ((250, 250), (60, 240), (240, 60), (150, 150))]
    s0 = pkg.synthetic.free_interior_cell_near(blocked, 30, 30)
    starts = [(float(s0[0]), float(s0[1]))] * 4
    paths, _ = pkg.cuda_api.batch_solve(layers, goals, starts)
    single, _ = _mars(pkg, n, n, seed=9)
    for (p, status), g, s in zip(paths, goals, starts):
        single.solve_total_cost([g])
        q, qs = single.extract_global_path(s[0], s[1], 0.4, *g)
        assert status == qs and p.shape == q.shape and np.max(np.abs(p[:, :2] - q[:, :2])) <= 1e-6


def test_plan_streamed_and_direct_delivery(pkg):
    import torch
    n = 1024
    cost = pkg.synthetic.smooth_cost_map(n, n, seed=13)
    d = cm.clearance(cost <= 0, *RMP[:2], 1.0)
    goal = pkg.synthetic.free_interior_cell_near((d <= RMP[0]).astype(np.float64), 700, 600)
    pinned_cost = torch.empty((n, n), dtype=torch.float64, pin_memory=True).numpy()
    pinned_cost[...] = cost
    a = pkg.cuda_api.DeviceLayer(n, n, 1.0, 0.1)
    a.set_obstacle_clearance(*RMP)
    assert a.plan_streamed(pinned_cost, goal)["converged"]
    b = pkg.cuda_api.DeviceLayer(n, n, 1.0, 0.1)
    b.set_cost_map(cost)
    b.set_obstacle_clearance(*RMP)
    out = torch.empty((n, n), dtype=torch.float64, pin_memory=True).numpy()
    assert b.set_total_cost_export(out, pkg.cuda_api.XFORM_INF_TO_MINUS1)
    assert b.solve_total_cost([goal])["converged"]
    b.synchronize()
    Tb = b.download_total_cost()
    assert np.array_equal(out, np.where(np.isinf(Tb), -1.0, Tb))
    assert np.array_equal(a.download_plane("ceff"), b.download_plane("ceff"))
    _same_T(a.download_total_cost(), Tb, 1e-13)


def test_time_stencils_leave_ceff(pkg):
    dev, _ = _mars(pkg, 500, 300, seed=6)
    C0, d0 = dev.download_plane("ceff"), dev.download_plane("clearance")
    dev.time_stencils()
    assert np.array_equal(dev.download_plane("ceff"), C0)
    assert np.array_equal(dev.download_plane("clearance"), d0)


def test_dd_solve_refuses_clearance(pkg):
    nx = 64
    strips = []
    for k in range(2):
        s = pkg.cuda_api.DeviceLayer(nx, 33, 1.0, 0.1)
        s.set_cost_map(np.ones((33, nx)))
        strips.append(s)
    strips[1].set_obstacle_clearance(*RMP)
    with pytest.raises(pkg.cuda_api.DymuError) as e:
        pkg.cuda_api.dd_solve(strips, [0, 32, 64], (10, 10))
    assert e.value.code == ERR_STATE


@pytest.mark.parametrize("bad", [(-1.0, 2.0, 1.0), (1.0, -2.0, 1.0), (1.0, 2.0, -1.0), (np.nan, 2.0, 1.0),
                                 (1.0, np.inf, 1.0), (0.0, 0.0, np.nan), (60.0, 69.0, 1.0)])
def test_argument_validation(pkg, bad):
    dev = pkg.cuda_api.DeviceLayer(64, 64, 1.0, 0.1)
    with pytest.raises(pkg.cuda_api.DymuError) as e:
        dev.set_obstacle_clearance(*bad)
    assert e.value.code == ERR_ARG
    dev.set_obstacle_clearance(60.0, 68.5, 1.0)  # R = 128 is accepted


# ---- 8. the planner class ------------------------------------------------------------------------
def test_class_goal_rules(pkg):
    assert pkg.planner_lib().lib.dymu_planner_set_obstacle_clearance(None, *RMP) == -1
    p = pkg.DyMuPathPlanner(1.0, 1.5, 2.0, pkg.planner_api.SWEEPING)
    assert not p.setObstacleClearance(*RMP)
    n = 64
    assert p.initGlobalLayer(1.0, 0.1, n, n)
    cost = np.ones((n, n))
    cost[32, 32] = 0.0
    assert p.setCostMap(cost)
    assert not p.setObstacleClearance(-1.0, 1.0, 1.0)
    assert p.setObstacleClearance(3.0, 4.0, 2.0)
    assert p.setGoal(34, 32)  # 2 m from the rock: inside the lethal ring
    assert not p.computeEntireTotalCostMap()
    assert not p.computeTotalCostMap(10, 10)
    assert p.setGoal(37, 32)  # 5 m: in the margin
    assert p.computeEntireTotalCostMap()
    assert p.computeTotalCostMap(10, 10)
    assert p.setObstacleClearance(0.0, 0.0, 0.0)
    assert p.setGoal(34, 32) and p.computeEntireTotalCostMap()


@pytest.mark.parametrize("approach", [0, 1])
def test_class_repair_scenario_with_clearance(pkg, approach):
    syn = pkg.synthetic
    n = 200
    p = sc.make_planner(pkg.DyMuPathPlanner, approach, n, n)
    assert p.setObstacleClearance(1.0, 2.0, 1.0)
    g = sc.global_scenario(p, syn, n, n, seed=42, entire=True)
    assert g["ok"] and len(g["path"]) > 10
    r = sc.repair_scenario(p, syn, g["path"])
    assert isinstance(r["repaired"], bool)
    if r["repaired"]:
        assert len(r["traj"]) > 0


def test_flat_c_view_of_the_reference(ref_lib):
    p = ref_lib.DyMuPathPlanner(1.0, 1.5, 2.0, 1)
    assert p.initGlobalLayer(1.0, 0.1, 32, 32)
    assert ref_lib.lib.dymu_planner_set_obstacle_clearance(p._h, *RMP) == -1
