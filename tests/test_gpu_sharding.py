"""Domain decomposition on the GPU: k logical strips on one device must reproduce the
single-grid solve (SURVEY.md section 4, 'multi-GPU without a cluster')."""
import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu

UNBOUNDED = 10**6   # a phase budget no strip exhausts: every strip converges before it trades rows


def test_batched_slots_advance_and_rows(pkg):
    """export/import round trip, then a solve_advance on the clean work list of a converged solve
    wakes the tiles of a row lowered by hand."""
    import torch
    api = pkg.cuda_api
    n = 128
    dev = api.DeviceLayer(n, n)
    dev.set_cost_map(np.ones((n, n)))
    dev.solve_total_cost([(64, 64)])
    T0 = dev.download_total_cost()
    row = torch.empty(n, dtype=torch.float64, device="cuda")
    dev.export_rows(10, 1, row.data_ptr(), True)
    assert np.array_equal(row.cpu().numpy(), T0[10])
    lower = torch.full((n,), 0.5, dtype=torch.float64, device="cuda")
    assert dev.import_rows_min_key(10, 1, lower.data_ptr(), True) == (True, 0.5)
    assert dev.import_rows_min_key(10, 1, lower.data_ptr(), True) == (False, float("inf"))
    assert dev.solve_advance([(9, 12)], 0.5, 1 << 20)["converged"]
    T1 = dev.download_total_cost()
    assert np.all(T1 <= T0) and T1[11, 5] == 1.5 and T1[10, 5] == 0.5


@pytest.mark.parametrize("phases", [1, 5, 40])
def test_phase_bounded_solve_equals_one_shot(pkg, phases):
    """dymu_solve_start + dymu_solve_advance in slices of `phases` solver phases reach the same
    fixed point as one dymu_solve_total_cost launch (the pending work lists survive between
    launches)."""
    api, syn = pkg.cuda_api, pkg.synthetic
    ny, nx = 416, 352
    cost = syn.smooth_cost_map(ny, nx, seed=8, obstacle_fraction=0.05)
    goal = syn.free_interior_cell_near(cost <= 0, 100, 300)
    dev = api.DeviceLayer(nx, ny)
    dev.set_cost_map(cost)
    one = dev.solve_total_cost([goal])
    T1 = dev.download_total_cost()
    st = dev.solve_start(goal, phases)
    launches, total_phases = 1, st["outer_iterations"]
    while not st["converged"]:
        assert st["outer_iterations"] == phases
        st = dev.solve_advance([], 0.0, phases)
        launches += 1
        total_phases += st["outer_iterations"]
        assert launches < 100000
    Tb = dev.download_total_cost()
    assert np.array_equal(np.isinf(Tb), np.isinf(T1))
    assert rel_err(Tb, T1) <= 1e-12
    if phases == 1:
        assert launches > 10
    # slicing must not change the schedule much: same order of magnitude of phases
    assert total_phases <= 2 * one["outer_iterations"] + 4
    # nothing pending any more: another advance is a no-op
    again = dev.solve_advance([], 0.0, phases)
    assert again["converged"] and again["tile_activations"] == 0


# goal row 180: the goal lies in an interior strip for k >= 3; goal row 40: in the first strip, so
# with an unbounded budget the converged front of one strip after the other crosses every cut
@pytest.mark.parametrize("k,phases,goal_row", [(2, 3, 180), (3, 8, 180), (4, 2, 180),
                                               (2, UNBOUNDED, 40), (3, UNBOUNDED, 40), (4, UNBOUNDED, 40)])
def test_pipelined_strips_equal_single_grid(pkg, k, phases, goal_row):
    import torch
    sh, api, syn = pkg.sharding, pkg.cuda_api, pkg.synthetic
    ny, nx = 384, 320
    cost = syn.smooth_cost_map(ny, nx, seed=21, obstacle_fraction=0.04)
    gi, gj = syn.free_interior_cell_near(cost <= 0, 200, goal_row)
    whole = api.DeviceLayer(nx, ny)
    whole.set_cost_map(cost)
    whole.solve_total_cost([(gi, gj)])
    T1 = whole.download_total_cost()
    strips = []
    for r in range(k):
        lay = sh.StripLayout(ny, k, r)
        strips.append(sh.CudaStrip(api, lay, nx, cost[lay.r0:lay.r1], 0, torch))
    rounds = sh.dd_solve_lockstep(strips, (gi, gj), phases_per_round=phases)
    Tk = np.vstack([s.own_rows() for s in strips])
    assert rounds >= 2
    assert np.array_equal(np.isinf(Tk), np.isinf(T1))
    assert rel_err(Tk, T1) <= 1e-12


def _strip_layers(pkg, cost, k, devices):
    """DeviceLayers of k row strips of `cost` (ghost rows = obstacles) + the cut rows."""
    sh, api = pkg.sharding, pkg.cuda_api
    ny, nx = cost.shape
    layers, cuts = [], [0]
    for r in range(k):
        lay = sh.StripLayout(ny, k, r)
        d = api.DeviceLayer(nx, lay.ny_local, 1.0, 0.1, device=devices[r % len(devices)])
        d.set_cost_map(lay.local_cost(cost[lay.r0:lay.r1]))
        layers.append((d, lay))
        cuts.append(lay.r1)
    return layers, cuts


def _gather_strips(layers):
    return np.vstack([d.download_total_cost()[lay.first_own:lay.last_own + 1] for d, lay in layers])


@pytest.mark.parametrize("k,phases", [(2, 8), (3, 32), (5, 2)])
def test_dd_solve_c_abi_on_one_device(pkg, k, phases):
    """dymu_dd_solve with k strips that all live on one GPU (one host thread per strip, rows copied
    device to device): same plane as the single-grid solve."""
    api, syn = pkg.cuda_api, pkg.synthetic
    ny, nx = 448, 352
    cost = syn.smooth_cost_map(ny, nx, seed=23, obstacle_fraction=0.04)
    goal = syn.free_interior_cell_near(cost <= 0, 120, 300)
    whole = api.DeviceLayer(nx, ny)
    whole.set_cost_map(cost)
    whole.solve_total_cost([goal])
    T1 = whole.download_total_cost()
    layers, cuts = _strip_layers(pkg, cost, k, [0])
    st = api.dd_solve([d for d, _ in layers], cuts, goal, phases)
    assert st["converged"] and st["rounds"] >= 2
    Tk = _gather_strips(layers)
    assert np.array_equal(np.isinf(Tk), np.isinf(T1))
    assert rel_err(Tk, T1) <= 1e-12
    # a second solve on the same contexts (other goal) starts clean
    goal2 = syn.free_interior_cell_near(cost <= 0, 300, 60)
    whole.solve_total_cost([goal2])
    api.dd_solve([d for d, _ in layers], cuts, goal2, phases)
    assert rel_err(_gather_strips(layers), whole.download_total_cost()) <= 1e-12


def test_dd_solve_c_abi_across_devices(pkg):
    """The same with every strip on its own GPU (peer copies over NVLink); skipped below 2 GPUs.
    16384^2 (BASELINE configs[4]) when the box has the memory for it, else 4096^2."""
    import torch
    ng = torch.cuda.device_count()
    if ng < 2:
        pytest.skip("needs at least two GPUs")
    api, syn = pkg.cuda_api, pkg.synthetic
    n, base = 16384, 4096
    tile = syn.smooth_cost_map(base, base, seed=20261018, obstacle_fraction=0.03)   # periodic fBm
    cost = np.tile(tile, (n // base, n // base))
    g0 = syn.free_interior_cell_near(tile <= 0, base // 2, base // 2)
    goal = (g0[0] + (n // base // 2) * base, g0[1] + (n // base // 2) * base)
    whole = api.DeviceLayer(n, n, device=0)
    whole.set_cost_map(cost)
    assert whole.solve_total_cost([goal])["converged"]
    T1 = whole.download_total_cost()
    whole.close()
    layers, cuts = _strip_layers(pkg, cost, ng, list(range(ng)))
    st = api.dd_solve([d for d, _ in layers], cuts, goal, 32)
    assert st["converged"]
    Tk = _gather_strips(layers)
    assert np.array_equal(np.isinf(Tk), np.isinf(T1))
    assert rel_err(Tk, T1) <= 1e-12


def test_batch_solve_c_abi(pkg):
    """dymu_batch_solve over two contexts (two GPUs if present, else both on GPU 0): every query's
    plane and path equal the single-context result."""
    import torch
    api, syn = pkg.cuda_api, pkg.synthetic
    n = 512
    cost = syn.smooth_cost_map(n, n, seed=4)
    ob = cost <= 0
    rng = np.random.default_rng(3)
    goals = [syn.free_interior_cell_near(ob, int(rng.uniform(0.1, 0.9) * n), int(rng.uniform(0.1, 0.9) * n))
             for _ in range(11)]
    starts = [syn.free_interior_cell_near(ob, int(rng.uniform(0.1, 0.9) * n), int(rng.uniform(0.1, 0.9) * n))
              for _ in range(11)]
    devs = [0, 1] if torch.cuda.device_count() >= 2 else [0, 0]
    layers = []
    for d in devs:
        L = api.DeviceLayer(n, n, device=d)
        L.set_cost_map(cost)
        L.reserve_slots(4)
        layers.append(L)
    paths, ms = api.batch_solve(layers, goals, [[float(a), float(b)] for a, b in starts], cap=4096)
    assert len(paths) == 11 and (ms > 0).all()
    one = api.DeviceLayer(n, n, device=0)
    one.set_cost_map(cost)
    for q in (0, 5, 10):
        one.solve_total_cost([goals[q]])
        w, status = one.extract_global_path(float(starts[q][0]), float(starts[q][1]), 0.4, goals[q][0], goals[q][1])
        got, gstatus = paths[q]
        assert gstatus == status and got.shape[0] == len(w)
        assert np.max(np.abs(got[:, :2] - w[:, :2])) <= 1e-9
