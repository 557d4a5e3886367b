"""GPU parity of the global layer through the device C ABI (include/dymu_cuda.h) against the
CPU oracle: cost-map stencils bit-exact, total-cost map <= 1e-9 relative (north_star bound;
observed ~1e-15), identical unreachable mask, waypoints <= 1e-3 cell."""
import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu

TOL_T = 1e-9      # relative, total-cost map (BASELINE.json north_star)
TOL_WP = 1e-3     # cells, waypoint positions


def _mars(pkg, oracle_mod, ny, nx, seed):
    syn = pkg.synthetic
    elev, terr = syn.mars_dem(ny, nx, seed=seed)
    lut, slopes, locs = syn.default_lut()
    po = oracle_mod.Port(1.0, 1.5, 2.0, oracle_mod.SWEEPING)
    po.initGlobalLayer(1.0, 0.1, nx, ny)
    assert po.computeCostMap(lut, slopes, locs, elev, terr)
    dev = pkg.cuda_api.DeviceLayer(nx, ny, 1.0, 0.1)
    dev.compute_cost_map(lut, slopes, len(locs), elev, terr)
    return po, dev


@pytest.mark.parametrize("ny,nx,seed", [(100, 100, 1), (129, 257, 2), (300, 300, 3), (64, 64, 4)])
def test_cost_map_stencils_bit_exact(pkg, oracle_mod, ny, nx, seed):
    po, dev = _mars(pkg, oracle_mod, ny, nx, seed)
    assert np.array_equal(dev.download_plane_u8("obstacle"), po.plane("isObstacle"))
    for name in ("slope", "raw_cost", "cost", "hazard_density", "trafficability"):
        a, b = dev.download_plane(name), po.plane(name)
        assert rel_err(a, b) <= 1e-14, name
    # second call exercises the smoothing quirk (seeded with the previous cost, G.cpp:299)
    syn = pkg.synthetic
    elev, terr = syn.mars_dem(ny, nx, seed=seed)
    lut, slopes, locs = syn.default_lut()
    po.computeCostMap(lut, slopes, locs, elev, terr)
    dev.compute_cost_map(lut, slopes, len(locs), elev, terr)
    assert rel_err(dev.download_plane("cost"), po.plane("cost")) <= 1e-14


@pytest.mark.parametrize("ny,nx,seed", [(100, 100, 1), (129, 257, 2), (300, 300, 3), (64, 64, 4),
                                        (33, 95, 5)])
def test_total_cost_map_matches_oracle(pkg, oracle_mod, ny, nx, seed):
    po, dev = _mars(pkg, oracle_mod, ny, nx, seed)
    ob = po.plane("isObstacle")
    gi, gj = pkg.synthetic.free_interior_cell_near(ob, nx // 2, ny // 2)
    assert po.setGoal(gi, gj) and po.computeEntireTotalCostMap()
    stats = dev.solve_total_cost([(gi, gj)])
    assert stats["converged"] == 1
    T = dev.download_total_cost()
    To = po.plane("total_cost")
    assert np.array_equal(np.isinf(T), np.isinf(To)), "unreachable mask differs"
    assert rel_err(T, To) <= TOL_T
    Tm = dev.download_total_cost(xform=pkg.cuda_api.XFORM_INF_TO_MINUS1)
    assert np.array_equal(Tm < 0, np.isinf(To))
    assert po.fixed_point_violations(T, 1e-12) == 0
    assert dev.count_reached() == int(np.isfinite(To).sum())


def test_set_cost_map_variant_and_path(pkg, oracle_mod):
    nx = ny = 200
    cost = pkg.synthetic.smooth_cost_map(ny, nx, seed=9)
    po = oracle_mod.Port(1.0, 1.5, 2.0, oracle_mod.SWEEPING)
    po.initGlobalLayer(1.0, 0.1, nx, ny)
    po.setCostMap(cost)
    dev = pkg.cuda_api.DeviceLayer(nx, ny, 1.0, 0.1)
    dev.set_cost_map(cost)
    ob = po.plane("isObstacle")
    assert np.array_equal(dev.download_plane_u8("obstacle"), ob)
    gi, gj = pkg.synthetic.free_interior_cell_near(ob, 160, 160)
    si, sj = pkg.synthetic.free_interior_cell_near(ob, 40, 40)
    po.setGoal(gi, gj)
    po.computeEntireTotalCostMap()
    dev.solve_total_cost([(gi, gj)])
    assert rel_err(dev.download_total_cost(), po.plane("total_cost")) <= TOL_T
    assert po.computeGlobalPath(float(si), float(sj)) == 1
    ref_path = po.current_path
    wps, status = dev.extract_global_path(float(si), float(sj), 0.4, gi, gj)
    assert status == 0
    assert wps.shape[0] == ref_path.shape[0] - 1  # goal waypoint is appended by the host
    assert np.max(np.abs(wps[:, :2] - ref_path[:-1, :2])) <= TOL_WP
    head = np.arctan2(-wps[:-1, 4], -wps[:-1, 3])
    assert np.max(np.abs(head - ref_path[1:-1, 3])) <= 1e-6


def test_batched_goals_share_one_launch(pkg, oracle_mod):
    nx = ny = 160
    cost = pkg.synthetic.smooth_cost_map(ny, nx, seed=11)
    dev = pkg.cuda_api.DeviceLayer(nx, ny, 1.0, 0.1)
    dev.set_cost_map(cost)
    dev.reserve_slots(4)
    ob = dev.download_plane_u8("obstacle")
    goals = [pkg.synthetic.free_interior_cell_near(ob, x, y) for x, y in
             ((30, 30), (120, 40), (80, 80), (40, 130))]
    dev.solve_total_cost(goals)
    starts = [[20.0, 140.0], [100.0, 100.0], [30.0, 30.0], [140.0, 25.0]]
    paths, status = dev.extract_global_path_batch([0, 1, 2, 3], starts, 0.4, goals)
    for q in range(4):
        single, st1 = dev.extract_global_path(starts[q][0], starts[q][1], 0.4, goals[q][0], goals[q][1],
                                              slot=q)
        assert status[q] == st1 and np.array_equal(paths[q], single, equal_nan=True)
    for q, (gi, gj) in enumerate(goals):
        po = oracle_mod.Port(1.0, 1.5, 2.0, 1)
        po.initGlobalLayer(1.0, 0.1, nx, ny)
        po.setCostMap(cost)
        po.setGoal(gi, gj)
        po.computeEntireTotalCostMap(heap=True)
        assert rel_err(dev.download_total_cost(slot=q), po.plane("total_cost")) <= TOL_T


def test_overlapped_total_cost_download(pkg):
    """dymu_download_total_cost_begin/_end around a path extraction deliver the same matrix
    as the synchronous getTotalCostMatrix read-back (inf -> -1, G.cpp:799-811)."""
    nx, ny = 200, 150
    dev = pkg.cuda_api.DeviceLayer(nx, ny, 1.0, 0.1)
    dev.set_cost_map(pkg.synthetic.smooth_cost_map(ny, nx, seed=5))
    ob = dev.download_plane_u8("obstacle")
    goal = pkg.synthetic.free_interior_cell_near(ob, 150, 100)
    dev.solve_total_cost([goal])
    want = dev.download_total_cost(xform=pkg.cuda_api.XFORM_INF_TO_MINUS1)
    got = np.full((ny, nx), np.nan)
    dev.download_total_cost_begin(got, xform=pkg.cuda_api.XFORM_INF_TO_MINUS1)
    wps, status = dev.extract_global_path(20.0, 20.0, 0.4, goal[0], goal[1])
    dev.download_total_cost_end()
    assert np.array_equal(got, want)
    assert status == 0 and len(wps) > 10
    # and the context keeps working afterwards
    # (two solves agree to rounding, not bit for bit: blocks of a tile read each other's cells
    # while they are being relaxed, and floating-point evaluation is not exactly monotone)
    dev.solve_total_cost([goal])
    again = dev.download_total_cost(xform=pkg.cuda_api.XFORM_INF_TO_MINUS1)
    assert np.array_equal(again < 0, want < 0) and rel_err(again, want) <= 1e-13


@pytest.mark.parametrize("goal_xy,first_phases", [((150, 300), 3), ((40, 20), 1), ((200, 590), 50)])
def test_streamed_plan_equals_upload_then_solve(pkg, goal_xy, first_phases):
    """dymu_plan_streamed (rows around the goal first, the rest opened while the solve is under
    way) reaches the fixed point of dymu_set_cost_map + dymu_solve_total_cost, twice in a row on
    different maps (the second call must not see anything of the first)."""
    nx, ny = 352, 608
    api, syn = pkg.cuda_api, pkg.synthetic
    for seed in (31, 32):
        cost = syn.smooth_cost_map(ny, nx, seed=seed, obstacle_fraction=0.0)
        plain = api.DeviceLayer(nx, ny)
        plain.set_cost_map(cost)
        goal = syn.free_interior_cell_near(plain.download_plane_u8("obstacle"), *goal_xy)
        plain.solve_total_cost([goal])
        want = plain.download_total_cost()
        if seed == 31:
            dev = api.DeviceLayer(nx, ny)
        st = dev.plan_streamed(np.ascontiguousarray(cost), goal, first_phases)
        assert st["converged"]
        got = dev.download_total_cost()
        assert np.array_equal(np.isinf(got), np.isinf(want))
        fin = np.isfinite(want) & (want > 0)
        assert np.max(np.abs(got[fin] - want[fin]) / want[fin]) <= 1e-13
        assert np.array_equal(dev.download_plane("ceff"), plain.download_plane("ceff"))


def test_abandoned_bounded_solve_leaves_no_stale_wakeups(pkg):
    """A phase-bounded solve that is abandoned leaves wake-up flags / keys of its pending tiles
    behind; the next full solve must not inherit them (a set flag would swallow that tile's
    wake-up and the kernel would report convergence with part of the plane unpropagated)."""
    n = 512
    cost = pkg.synthetic.smooth_cost_map(n, n, seed=5)
    ob = cost <= 0
    ga = pkg.synthetic.free_interior_cell_near(ob, 100, 120)
    gb = pkg.synthetic.free_interior_cell_near(ob, 400, 380)
    clean = pkg.cuda_api.DeviceLayer(n, n)
    clean.set_cost_map(cost)
    assert clean.solve_total_cost([gb])["converged"]
    want = clean.download_total_cost()
    dut = pkg.cuda_api.DeviceLayer(n, n)
    dut.set_cost_map(cost)
    st = dut.solve_start(ga, 3)
    assert not st["converged"]
    assert dut.solve_total_cost([gb])["converged"]          # abandons the pending lists
    got = dut.download_total_cost()
    assert np.array_equal(np.isinf(got), np.isinf(want))
    fin = np.isfinite(want) & (want > 0)
    assert np.max(np.abs(got[fin] - want[fin]) / want[fin]) <= 1e-13
    # the same after reset_total_cost() dropped the pending work of a phase-bounded solve
    st = dut.solve_start(ga, 2)
    dut.reset_total_cost()
    assert dut.solve_total_cost([gb])["converged"]
    got = dut.download_total_cost()
    assert np.max(np.abs(got[fin] - want[fin]) / want[fin]) <= 1e-13


def test_two_contexts_on_two_devices_from_one_thread(pkg):
    """Every entry point selects its context's device itself (and restores the caller's)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    n = 256
    cost = pkg.synthetic.smooth_cost_map(n, n, seed=9)
    goal = pkg.synthetic.free_interior_cell_near(cost <= 0, 128, 128)
    torch.cuda.set_device(0)
    a = pkg.cuda_api.DeviceLayer(n, n, device=0)
    b = pkg.cuda_api.DeviceLayer(n, n, device=1)
    assert torch.cuda.current_device() == 0
    out = []
    for d in (a, b, a, b):          # interleaved use from one host thread
        d.set_cost_map(cost)
        assert d.solve_total_cost([goal])["converged"]
        out.append(d.download_total_cost())
    assert torch.cuda.current_device() == 0
    fin = np.isfinite(out[0]) & (out[0] > 0)
    for T in out[1:]:
        assert np.max(np.abs(T[fin] - out[0][fin]) / out[0][fin]) <= 1e-13


def test_incremental_resolve_equals_full_solve(pkg):
    """dymu_solve_incremental after raising and lowering trafficability / hazard_density on patches
    of global nodes (what a local repair feeds back, L.cpp:264-274, 388-394): same plane as a solve
    from scratch, with only a part of the map invalidated."""
    n = 768
    syn, api = pkg.synthetic, pkg.cuda_api
    cost = syn.smooth_cost_map(n, n, seed=12)
    goal = syn.free_interior_cell_near(cost <= 0, 600, 560)
    dev, ref = api.DeviceLayer(n, n), api.DeviceLayer(n, n)
    dev.set_cost_map(cost)
    ref.set_cost_map(cost)
    st, inv = dev.solve_incremental(goal)
    assert st["converged"] and inv is None                      # nothing resident yet: full solve
    st, inv = dev.solve_incremental(goal)
    assert st["converged"] and inv == 0 and st["tile_activations"] == 0   # nothing changed
    rng = np.random.default_rng(2)
    for step in range(3):
        for d in (dev, ref):
            r = np.random.default_rng(100 + step)
            for _ in range(3):
                i0, j0 = int(r.integers(40, 300)), int(r.integers(40, 300))
                w, h = int(r.integers(3, 30)), int(r.integers(3, 30))
                d.write_rect("trafficability", i0, j0, np.full((h, w), r.uniform(0.2, 0.9)))
                i0, j0 = int(r.integers(40, 700)), int(r.integers(40, 700))
                d.write_rect("hazard_density", i0, j0, np.full((4, 4), r.uniform(0.1, 0.6)))
            if step == 2:   # costs going down again
                d.write_rect("trafficability", 50, 50, np.ones((200, 200)))
        st, inv = dev.solve_incremental(goal)
        assert st["converged"] and inv is not None and 0 < inv < 0.25 * n * n, (step, inv)
        full = ref.solve_total_cost([goal])
        assert st["cell_updates"] < full["cell_updates"]
        T, Tf = dev.download_total_cost(), ref.download_total_cost()
        assert np.array_equal(np.isinf(T), np.isinf(Tf))
        fin = np.isfinite(Tf) & (Tf > 0)
        assert np.max(np.abs(T[fin] - Tf[fin]) / Tf[fin]) <= 1e-12, step
    # another goal: not reusable, full solve
    goal2 = syn.free_interior_cell_near(cost <= 0, 100, 100)
    st, inv = dev.solve_incremental(goal2)
    assert inv is None and st["converged"]
    ref.solve_total_cost([goal2])
    T, Tf = dev.download_total_cost(), ref.download_total_cost()
    fin = np.isfinite(Tf) & (Tf > 0)
    assert np.array_equal(np.isinf(T), np.isinf(Tf)) and np.max(np.abs(T[fin] - Tf[fin]) / Tf[fin]) <= 1e-13


@pytest.mark.parametrize("ny,nx,streamed", [(777, 1000, False), (608, 352, True), (64, 64, False)])
def test_direct_delivery_of_total_cost_matrix(pkg, ny, nx, streamed):
    """dymu_set_total_cost_export: the solve kernel stores every tile of the total-cost matrix into
    the caller's page-locked buffer once the front is past it.  What arrives is, bit for bit, what a
    read-back of the plane gives afterwards (inf -> -1, G.cpp:799-811); columns beyond nx are not
    touched; an unpinned buffer is declined and the ordinary read-back keeps working."""
    import torch
    api, syn = pkg.cuda_api, pkg.synthetic
    dev = api.DeviceLayer(nx, ny)
    cost = np.ascontiguousarray(syn.smooth_cost_map(ny, nx, seed=11))
    dev.set_cost_map(cost)
    ob = dev.download_plane_u8("obstacle")
    goal = syn.free_interior_cell_near(ob, nx // 3, ny // 2)
    ld = nx + 5
    pinned = torch.full((ny, ld), float("nan"), dtype=torch.float64).pin_memory()
    buf = pinned.numpy()
    assert dev.set_total_cost_export(buf, xform=api.XFORM_INF_TO_MINUS1)
    n_tiles = ((nx + 31) // 32) * ((ny + 31) // 32)
    for rep in range(2):  # the second solve must not take anything of the first for delivered
        buf[:] = np.nan
        st = dev.plan_streamed(cost, goal) if streamed else dev.solve_total_cost([goal])
        assert st["converged"]
        assert st["tiles_delivered_early"] + st["tiles_delivered_late"] >= n_tiles
        if nx * ny > 100000:
            assert st["tiles_delivered_early"] > n_tiles // 2, st
        # same pointer, ld and transform: nothing left to copy
        dev.download_total_cost_begin(buf, xform=api.XFORM_INF_TO_MINUS1)
        dev.download_total_cost_end()
        want = np.empty((ny, nx))
        dev.download_total_cost(out=want, xform=api.XFORM_INF_TO_MINUS1)
        assert np.array_equal(buf[:, :nx], want)
        assert np.isnan(buf[:, nx:]).all()
    # a change to the plane ends the "already delivered" state: the copy happens again
    dev.write_rect("total_cost", goal[0], goal[1], np.array([[123.0]]))
    dev.download_total_cost_begin(buf, xform=api.XFORM_INF_TO_MINUS1)
    dev.download_total_cost_end()
    assert buf[goal[1], goal[0]] == 123.0 and np.isnan(buf[:, nx:]).all()
    # switched off: solves leave the buffer alone
    dev.set_total_cost_export(None)
    buf[:] = np.nan
    dev.solve_total_cost([goal])
    assert np.isnan(buf).all()
    # pageable memory is declined, not an error
    plain = np.empty((ny, nx))
    assert dev.set_total_cost_export(plain, xform=api.XFORM_INF_TO_MINUS1) is False
    dev.solve_total_cost([goal])
    dev.download_total_cost(out=plain, xform=api.XFORM_INF_TO_MINUS1)
    # (two solves agree to rounding, not bit for bit)
    assert np.array_equal(plain < 0, want < 0) and rel_err(plain, want) <= 1e-13
